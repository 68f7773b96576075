// smooth.cu -- keypoint smoothing across video frames (ekp_smooth_humans): a One Euro filter (Casiez, Roussel, Vogel,
// CHI 2012) per track id, part and axis, on the device human tables and the tracker's ids.
//
// Specification (include/ekpose_b200.h, "smoothing").  Image i of a call is frame i % F of sequence i / F.  Row p of a
// frame with id = ids[p] >= 0 uses its sequence's entry of that id; a frame first resolves every row whose id has an
// entry, then opens entries for the others in row order (in a free entry, else in the one with the smallest
// (last_seen, id) not seen in this frame: common.cuh's evict_first); entries expire as the tracker's tracks do
// (common.cuh's expired).  Per present part and axis the entry's filter takes the raw coordinate in float64, +-*/ and
// fabs only, each rounded (-fmad=false here, -ffp-contract=off on the host).
//
// One CTA per sequence, over chunks of at most `chunk` frames:
//   1. one warp resolves every (frame, row) of the chunk to an entry, walking the frames in order over shared-memory
//      tables of the entries' (tag, last_seen), a compact list of the live entries and a stack of the free ones.  It
//      records, per frame and entry, the row that used the entry (and whether it opened it) in an inverse map, and lists
//      the entries the chunk touched.  The other warps meanwhile write every output of the chunk as the raw coordinate
//      (present parts of rows < num_humans) or 0: rows that pass through (id < 0) keep that;
//   2. after a barrier, one thread per (touched entry, part, axis) walks the chunk's frames on its own, with the filter
//      values in registers (restarting at a birth in its entry), and overwrites the outputs of its rows.
// No barrier sits inside the float64 arithmetic, and the filter values (too many for shared memory at 512 entries) are
// read and written once per chunk from the caller's state.
// The whole of it is __host__ __device__: ekp_debug_smooth_host runs the same code with one thread on the CPU (a test
// hook, not a CPU path of ekp_smooth_humans), where a warp is one lane and the barriers are no-ops.  Entry indices are
// not observable (lookups go by id, eviction ties by id), so the entry a birth takes need not match between the two.
#include <math.h>

#include <vector>

#include "common.cuh"

namespace ekp {

#define HD __host__ __device__ __forceinline__

static const int kComp = 2 * EKP_NUM_PART;         // (part, axis) components of an entry
static const int kSmoothThreads = 512;
static const size_t kInvBytes = 64 * 1024;         // the inverse map of a chunk: chunk x max_tracks uint16
static const unsigned short kNone = 0xFFFF;        // inverse map: the entry is not used in that frame
static const unsigned short kBirth = 0x8000;       // ... used by the row in the low bits, which opened it
static const double kPi = 3.141592653589793;       // the double nearest pi

struct SmoothHead { int frame, pad0, pad1, pad2; };  // frames seen, per sequence
struct SmoothEntry { unsigned tag; int last_seen; }; // tag = id + 1 (0: free); frame of the last use
static_assert(sizeof(SmoothHead) == 16 && sizeof(SmoothEntry) == 8, "state layout");

// per sequence: the head, the entries, then per (entry, component) xh, dxh (float64) and the frame of the last sample
// (int, -1: none).  8-byte multiple, so every sequence's float64 arrays stay aligned.
HD size_t smooth_seq_bytes(int max_tracks) {
    return sizeof(SmoothHead) + (sizeof(SmoothEntry) + (2 * sizeof(double) + sizeof(int)) * kComp) * (size_t) max_tracks;
}
size_t smooth_state_seq_bytes(int max_tracks) { return smooth_seq_bytes(max_tracks); }

HD void sbar() {
#ifdef __CUDA_ARCH__
    __syncthreads();
#endif
}
HD void wsync() {
#ifdef __CUDA_ARCH__
    __syncwarp();
#endif
}
HD unsigned wballot(bool pred) {
#ifdef __CUDA_ARCH__
    return __ballot_sync(~0u, pred);
#else
    return pred ? 1u : 0u;
#endif
}
HD int popc(unsigned v) {
#ifdef __CUDA_ARCH__
    return __popc(v);
#else
    return __builtin_popcount(v);
#endif
}
HD int ctz(unsigned v) {   // v != 0
#ifdef __CUDA_ARCH__
    return __ffs(v) - 1;
#else
    return __builtin_ctz(v);
#endif
}

struct SmoothArgs {
    const int* num_humans;   // [n]
    const ekp_peak* parts;   // [n][max_humans][18]
    const int* ids;          // [n][max_humans]
    int max_humans, F, max_tracks, max_age, chunk;
    double fps, min_cutoff, beta, tau_d;   // tau_d = 1 / ((2 pi) d_cutoff)
    float* xy;               // [n][max_humans][18][2]
    unsigned char* state;    // [n_seq] x smooth_seq_bytes(max_tracks)
};

// one sequence's working set (shared memory on the device)
struct SmoothWork {
    unsigned* etag;          // [max_tracks] entry tags
    int* eseen;              // [max_tracks] entry last_seen
    int* live;               // [max_tracks] the live entries
    int* freest;             // [max_tracks] the free entries (a stack)
    int* tlist;              // [max_tracks] the entries the chunk touched
    int* rowent;             // [max_humans] per row of the frame: its entry, -1 passed through, -2 to open
    int* cnt;                // [4] touched entries
    unsigned char* touch;    // [max_tracks]
    unsigned short* inv;     // [chunk][max_tracks]
};

// Carves the working set out of `base` (nullptr: only sizes it); returns its bytes.
HD size_t smooth_work_layout(int max_humans, int max_tracks, int chunk, unsigned char* base, SmoothWork* w) {
    size_t off = 0;
    auto take = [&](size_t bytes) { unsigned char* p = base ? base + off : nullptr; off += (bytes + 15) & ~(size_t) 15; return p; };
    SmoothWork t;
    t.etag = (unsigned*) take(sizeof(unsigned) * max_tracks);
    t.eseen = (int*) take(sizeof(int) * max_tracks);
    t.live = (int*) take(sizeof(int) * max_tracks);
    t.freest = (int*) take(sizeof(int) * max_tracks);
    t.tlist = (int*) take(sizeof(int) * max_tracks);
    t.rowent = (int*) take(sizeof(int) * max_humans);
    t.cnt = (int*) take(sizeof(int) * 4);
    t.touch = (unsigned char*) take(max_tracks);
    t.inv = (unsigned short*) take(sizeof(unsigned short) * (size_t) chunk * max_tracks);
    if (w) *w = t;
    return off;
}

// frames per chunk: the inverse map takes at most kInvBytes
HD int smooth_chunk(int F, int max_tracks) {
    const int cap = (int) (kInvBytes / (sizeof(unsigned short) * max_tracks));
    return F < cap ? F : cap;
}

// One filter step at a sample x that follows the last one by g frames: the header's operations, in its order.
HD void one_euro_step(double x, int g, const SmoothArgs& A, double& xh, double& dxh) {
    const double te = (double) g / A.fps;
    const double a_d = 1.0 / (1.0 + A.tau_d / te);
    const double dx = (x - xh) / te;
    dxh = a_d * dx + (1.0 - a_d) * dxh;
    const double c = A.min_cutoff + A.beta * fabs(dxh);
    const double tau = 1.0 / ((2.0 * kPi) * c);
    const double a = 1.0 / (1.0 + tau / te);
    xh = a * x + (1.0 - a) * xh;
}

// Phase 1 of frames c0 .. c0 + FC - 1 on the `lanes` lanes of one warp.  nl / nf: live and free counts, warp-uniform.
HD void resolve_chunk(const SmoothArgs& A, int seq, const SmoothWork& W, int f0, int c0, int FC, int lane, int lanes, int& nl, int& nf) {
    const int MH = A.max_humans, MT = A.max_tracks;
    const unsigned below = (1u << lane) - 1u;
    for (int t = 0; t < FC; t++) {
        const int f = f0 + c0 + t, img = seq * A.F + c0 + t;
        const int P = min(max(A.num_humans[img], 0), MH);
        const int* idrow = A.ids + (size_t) img * MH;
        unsigned short* inv = W.inv + (size_t) t * MT;
        // expiry: compact the live list, push the expired entries on the free stack
        int kept = 0, freed = nf;
        for (int b = 0; b < nl; b += lanes) {
            const int k = b + lane;
            const int e = k < nl ? W.live[k] : -1;
            const bool keep = e >= 0 && !expired(W.eseen[e], f, A.max_age), drop = e >= 0 && !keep;
            const unsigned bk = wballot(keep), bd = wballot(drop);
            wsync();
            if (keep) W.live[kept + popc(bk & below)] = e;
            if (drop) { W.freest[freed + popc(bd & below)] = e; W.etag[e] = 0; }
            kept += popc(bk); freed += popc(bd);
            wsync();
        }
        nl = kept; nf = freed;
        // lookup of every row whose id has an entry: the lanes scan the live list together
        for (int p = 0; p < P; p++) {
            const int id = idrow[p];
            int r = -1;
            if (id >= 0) {
                r = -2;
                const unsigned tag = (unsigned) id + 1u;
                for (int b = 0; b < nl; b += lanes) {
                    const int k = b + lane;
                    const unsigned hit = wballot(k < nl && W.etag[W.live[k]] == tag);
                    if (hit) { r = W.live[b + ctz(hit)]; break; }   // warp-uniform
                }
            }
            if (lane == 0) W.rowent[p] = r;
        }
        wsync();
        for (int p = lane; p < P; p += lanes) {
            const int e = W.rowent[p];
            if (e >= 0) { W.eseen[e] = f; inv[e] = (unsigned short) p; W.touch[e] = 1; }
        }
        wsync();
        // births in row order
        for (int p = 0; p < P; p++) {
            if (W.rowent[p] != -2) continue;   // warp-uniform
            int e = -1;
            if (nf > 0) {
                e = W.freest[--nf];
                wsync();
                if (lane == 0) W.live[nl] = e;
                nl++;
            } else {   // the live entry of the smallest (last_seen, id) not seen in this frame
                int bs = 0, bid = 0;
                for (int k = lane; k < nl; k += lanes) {
                    const int q = W.live[k], s = W.eseen[q], id = (int) (W.etag[q] - 1u);
                    if (s != f && (e < 0 || evict_first(s, id, bs, bid))) { e = q; bs = s; bid = id; }
                }
#ifdef __CUDA_ARCH__
                for (int o = 16; o > 0; o >>= 1) {
                    const int oe = __shfl_xor_sync(~0u, e, o), os = __shfl_xor_sync(~0u, bs, o), oid = __shfl_xor_sync(~0u, bid, o);
                    if (oe >= 0 && (e < 0 || evict_first(os, oid, bs, bid))) { e = oe; bs = os; bid = oid; }
                }
#endif
            }
            if (e >= 0 && lane == 0) {   // e < 0 only for duplicate ids: the row passes through
                W.etag[e] = (unsigned) idrow[p] + 1u;
                W.eseen[e] = f;
                inv[e] = (unsigned short) (kBirth | p);
                W.touch[e] = 1;
            }
            wsync();
        }
    }
    // the entries the chunk touched, in entry order
    int nt = 0;
    for (int b = 0; b < MT; b += lanes) {
        const int e = b + lane;
        const bool on = e < MT && W.touch[e];
        const unsigned bt = wballot(on);
        if (on) { W.tlist[nt + popc(bt & below)] = e; W.touch[e] = 0; }
        nt += popc(bt);
    }
    if (lane == 0) W.cnt[0] = nt;
}

// Every output of frames c0 .. c0 + FC - 1, element u0, u0 + step, ...: the raw coordinate or 0.
HD void fill_chunk(const SmoothArgs& A, int seq, int c0, int FC, int u0, int step) {
    const int MH = A.max_humans, per = MH * EKP_NUM_PART;
    for (int u = u0; u < FC * per; u += step) {
        const int t = u / per, r = u - t * per, p = r / EKP_NUM_PART;
        const int img = seq * A.F + c0 + t;
        const size_t at = (size_t) img * per + r;
        const ekp_peak pk = A.parts[at];
        const bool on = p < min(max(A.num_humans[img], 0), MH) && pk.id >= 0;
        A.xy[2 * at] = on ? (float) (double) pk.x : 0.0f;
        A.xy[2 * at + 1] = on ? (float) (double) pk.y : 0.0f;
    }
}

// Phase 2: the filters of the touched entries over frames c0 .. c0 + FC - 1, item u0, u0 + step, ...
HD void filter_chunk(const SmoothArgs& A, int seq, const SmoothWork& W, double* gxh, double* gdxh, int* gfl, int f0, int c0,
                     int FC, int u0, int step) {
    const int MH = A.max_humans, MT = A.max_tracks, items = W.cnt[0] * kComp;
    for (int u = u0; u < items; u += step) {
        const int e = W.tlist[u / kComp], c = u % kComp, part = c >> 1, ax = c & 1;
        const size_t k = (size_t) e * kComp + c;
        double xh = gxh[k], dxh = gdxh[k];
        int fl = gfl[k];
        for (int t = 0; t < FC; t++) {
            const unsigned code = W.inv[(size_t) t * MT + e];
            if (code == kNone) continue;
            if (code & kBirth) fl = -1;
            const int p = (int) (code & ~(unsigned) kBirth);
            const size_t at = ((size_t) (seq * A.F + c0 + t) * MH + p) * EKP_NUM_PART + part;
            const ekp_peak pk = A.parts[at];
            if (pk.id < 0) continue;
            const double x = (double) (ax ? pk.y : pk.x);
            const int f = f0 + c0 + t;
            if (fl < 0) { xh = x; dxh = 0.0; }
            else one_euro_step(x, f - fl, A, xh, dxh);
            fl = f;
            A.xy[2 * at + ax] = (float) xh;
        }
        gxh[k] = xh; gdxh[k] = dxh; gfl[k] = fl;
    }
}

// Runs the F frames of sequence `seq` on thread `tid` of `nt` (nt % 32 == 0, or nt == 1 on the host).
HD void smooth_sequence(const SmoothArgs& A, int seq, const SmoothWork& W, int tid, int nt) {
    const int MT = A.max_tracks;
    unsigned char* base = A.state + smooth_seq_bytes(MT) * (size_t) seq;
    SmoothHead* gh = reinterpret_cast<SmoothHead*>(base);
    SmoothEntry* gent = reinterpret_cast<SmoothEntry*>(gh + 1);
    double* gxh = reinterpret_cast<double*>(gent + MT);
    double* gdxh = gxh + (size_t) MT * kComp;
    int* gfl = reinterpret_cast<int*>(gdxh + (size_t) MT * kComp);
    const int f0 = gh->frame;
    const int lanes = nt >= 32 ? 32 : 1, lane = tid % lanes;
    const bool resolver = tid < lanes;
    for (int k = tid; k < MT; k += nt) { W.etag[k] = gent[k].tag; W.eseen[k] = gent[k].last_seen; W.touch[k] = 0; }
    sbar();
    int nl = 0, nf = 0;   // meaningful in the resolving warp only
    if (resolver) {
        const unsigned below = (1u << lane) - 1u;
        for (int b = 0; b < MT; b += lanes) {
            const int k = b + lane;
            const bool on = k < MT && W.etag[k] != 0u, fr = k < MT && W.etag[k] == 0u;
            const unsigned bl = wballot(on), bf = wballot(fr);
            if (on) W.live[nl + popc(bl & below)] = k;
            if (fr) W.freest[nf + popc(bf & below)] = k;
            nl += popc(bl); nf += popc(bf);
        }
    }
    for (int c0 = 0; c0 < A.F; c0 += A.chunk) {
        const int FC = min(A.chunk, A.F - c0);
        for (int u = tid; u < FC * MT; u += nt) W.inv[u] = kNone;
        sbar();
        if (resolver) resolve_chunk(A, seq, W, f0, c0, FC, lane, lanes, nl, nf);
        if (nt == 1) fill_chunk(A, seq, c0, FC, 0, 1);
        else if (!resolver) fill_chunk(A, seq, c0, FC, tid - lanes, nt - lanes);
        sbar();
        filter_chunk(A, seq, W, gxh, gdxh, gfl, f0, c0, FC, tid, nt);
        sbar();
    }
    for (int k = tid; k < MT; k += nt) { gent[k].tag = W.etag[k]; gent[k].last_seen = W.eseen[k]; }
    if (tid == 0) gh->frame = f0 + A.F;
}

__global__ void __launch_bounds__(kSmoothThreads, 1) smooth_kernel(const SmoothArgs A) {
    extern __shared__ __align__(16) unsigned char smem[];
    SmoothWork W;
    smooth_work_layout(A.max_humans, A.max_tracks, A.chunk, smem, &W);
    smooth_sequence(A, blockIdx.x, W, threadIdx.x, blockDim.x);
}

// the largest working set: max_humans = max_tracks = EKP_LIMIT_TRACKS and a full inverse map
cudaError_t configure_smooth() {
    const size_t most = smooth_work_layout(EKP_LIMIT_TRACKS, EKP_LIMIT_TRACKS, smooth_chunk(1 << 30, EKP_LIMIT_TRACKS), nullptr, nullptr);
    return raise_dynamic_smem_limit(smooth_kernel, most);
}

static SmoothArgs smooth_args(const int* num_humans, const ekp_peak* parts, const int* ids, int n, int max_humans, void* state,
                              int n_seq, int max_tracks, int max_age, double fps, double min_cutoff, double beta, double d_cutoff,
                              float* xy) {
    const int F = n / n_seq;
    return SmoothArgs{num_humans, parts, ids, max_humans, F, max_tracks, max_age, smooth_chunk(F, max_tracks), fps, min_cutoff,
                      beta, 1.0 / ((2.0 * kPi) * d_cutoff), xy, static_cast<unsigned char*>(state)};
}

cudaError_t launch_smooth(const int* num_humans, const ekp_peak* parts, const int* ids, int n, int max_humans, void* state, int n_seq,
                          int max_tracks, int max_age, double fps, double min_cutoff, double beta, double d_cutoff, float* xy,
                          cudaStream_t stream) {
    const SmoothArgs A = smooth_args(num_humans, parts, ids, n, max_humans, state, n_seq, max_tracks, max_age, fps, min_cutoff, beta,
                                     d_cutoff, xy);
    const size_t smem = smooth_work_layout(max_humans, max_tracks, A.chunk, nullptr, nullptr);
    smooth_kernel<<<n_seq, kSmoothThreads, smem, stream>>>(A);
    return cudaGetLastError();
}

void debug_smooth_host(const int* num_humans, const ekp_peak* parts, const int* ids, int n, int max_humans, void* state, int n_seq,
                       int max_tracks, int max_age, double fps, double min_cutoff, double beta, double d_cutoff, float* xy) {
    const SmoothArgs A = smooth_args(num_humans, parts, ids, n, max_humans, state, n_seq, max_tracks, max_age, fps, min_cutoff, beta,
                                     d_cutoff, xy);
    std::vector<double> buf(smooth_work_layout(max_humans, max_tracks, A.chunk, nullptr, nullptr) / sizeof(double) + 2);
    SmoothWork W;
    smooth_work_layout(max_humans, max_tracks, A.chunk, reinterpret_cast<unsigned char*>(buf.data()), &W);
    for (int s = 0; s < n_seq; s++) smooth_sequence(A, s, W, 0, 1);
}

}  // namespace ekp
