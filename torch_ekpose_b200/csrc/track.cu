// track.cu -- stable person ids across video frames (ekp_track_humans): greedy one-to-one matching of each frame's
// people to the live tracks of its sequence by COCO's object keypoint similarity (OKS), on the device human tables.
//
// Specification (include/ekpose_b200.h, DESIGN.md section 8).  Image i of a call is frame i % F of sequence i / F.  The
// people of a frame are rows 0 .. min(num_humans, max_humans) - 1 of its part table; person p's similarity to live
// track t is the OKS in float64 with t's last pose as the ground truth (COCO keypoint j = reference part ORDER_COCO[j],
// pycocotools' sigmas and variances, area = the integer bounding-box area of t's present COCO parts, sum of exp(-e_j) in
// j order over the parts present in both, over their count; 0 when there are none).  Pairs with sim >= min_oks are
// accepted greedily in the total order (sim descending, track id ascending, row ascending); unmatched people open new
// tracks in row order, taking the sequence's next ids; a track last matched at frame f0 can be matched up to frame
// f0 + max_age + 1 and is dropped after that; a new track that finds every slot live takes the slot of the unmatched
// live track with the smallest (last_seen, id).
//
// One CTA per sequence walks its F frames in order (frame t needs the tracks frame t - 1 left); the sequence's tracks stay
// in shared memory for the whole call and go back to the caller's state buffer at the end.  Within a frame every phase
// is a thread-strided loop between barriers:
//   1. stage the people's COCO poses, drop expired tracks, list the live and the free slots;
//   2. every (person, live track) similarity into a shared-memory matrix (a frame whose P x L pairs do not fit it uses
//      a max_tracks x max_tracks scratch the state holds per sequence instead);
//   3. greedy matching in rounds: every free person picks its best free track, every free track its best free person
//      (each in the total order above; one warp per choice), and the mutual picks are accepted.  Such a pair is the first in the total order
//      of all pairs sharing its person or its track, so the serial greedy walk accepts it too, and removing it leaves the
//      greedy walk of the rest unchanged: the rounds give exactly the walk's matching, with no sort and no pair list;
//   4. matched tracks take their person's pose; unmatched people open tracks in row order, in free slots first, then in
//      the slots of the oldest unmatched tracks.
// The whole of it is __host__ __device__: ekp_debug_track_host runs the same code with one thread on the CPU (a test
// hook, not a CPU path of ekp_track_humans), where the barriers are no-ops and the shared-memory atomics plain
// increments.  Slot order is not observable (ties are broken by track id), so the atomically built slot lists need not be
// deterministic.
#include <math.h>
#include <string.h>

#include <vector>

#include "common.cuh"

namespace ekp {

#define HD __host__ __device__ __forceinline__

static const int kCoco = 17;
static const int kTrackThreads = 256;
static const size_t kTrackSmemMax = 227 * 1024;  // opt-in shared memory of one block on sm_100a (232,448 bytes)

struct TrackHead { int frame, next_id, pad0, pad1; };  // frames seen and the next id, per sequence
struct TrackSlot {       // 160 bytes
    int tag;             // track id + 1; 0 = free slot
    int last_seen;       // frame of the last match (or of the birth)
    unsigned mask;       // bit j: COCO keypoint j present in the last pose
    int pad;
    double area;         // integer bounding-box area of the present keypoints (1 when there are none)
    int xy[2 * kCoco];   // the last pose, map pixels
};
struct PersonPose {      // 152 bytes: one person of the current frame, as a TrackSlot holds it
    unsigned mask;
    int pad;
    double area;
    int xy[2 * kCoco];
};
static_assert(sizeof(TrackSlot) == 160 && sizeof(PersonPose) == 152, "state layout");

// per sequence: the head, the track slots, then a max_tracks x max_tracks scratch of similarities for frames whose
// similarity matrix does not fit the shared-memory cache (max_humans <= max_tracks)
HD size_t slots_bytes(int max_tracks) { return sizeof(TrackHead) + sizeof(TrackSlot) * (size_t) max_tracks; }
HD size_t seq_bytes(int max_tracks) { return slots_bytes(max_tracks) + sizeof(double) * (size_t) max_tracks * max_tracks; }
size_t track_seq_bytes(int max_tracks) { return seq_bytes(max_tracks); }

HD void bar() {
#ifdef __CUDA_ARCH__
    __syncthreads();
#endif
}
HD int bar_or(int pred) {
#ifdef __CUDA_ARCH__
    return __syncthreads_or(pred);
#else
    return pred;
#endif
}
HD int claim(int* counter) {
#ifdef __CUDA_ARCH__
    return atomicAdd(counter, 1);
#else
    return (*counter)++;
#endif
}

// COCO keypoint j = reference part ORDER_COCO[j] (torch_ekpose_b200/coco.py)
__constant__ const signed char kOrderCocoDev[kCoco] = {0, 15, 14, 17, 16, 5, 2, 6, 3, 7, 4, 11, 8, 12, 9, 13, 10};
[[maybe_unused]] static const signed char kOrderCocoHost[kCoco] = {0, 15, 14, 17, 16, 5, 2, 6, 3, 7, 4, 11, 8, 12, 9, 13, 10};
HD int coco_part(int j) {
#ifdef __CUDA_ARCH__
    return kOrderCocoDev[j];
#else
    return kOrderCocoHost[j];
#endif
}

// the COCO pose of one row of a part table (ekp_peak [18]: id -1 = absent)
HD void load_pose(const ekp_peak* row, PersonPose& out) {
    unsigned mask = 0;
    int x0 = 0, x1 = 0, y0 = 0, y1 = 0;
    for (int j = 0; j < kCoco; j++) {
        const ekp_peak pk = row[coco_part(j)];
        const bool on = pk.id >= 0;
        out.xy[2 * j] = on ? pk.x : 0;
        out.xy[2 * j + 1] = on ? pk.y : 0;
        if (on) {
            x0 = mask ? min(x0, pk.x) : pk.x; x1 = mask ? max(x1, pk.x) : pk.x;
            y0 = mask ? min(y0, pk.y) : pk.y; y1 = mask ? max(y1, pk.y) : pk.y;
            mask |= 1u << j;
        }
    }
    out.mask = mask;
    out.area = mask ? (double) (((long long) x1 - x0 + 1) * ((long long) y1 - y0 + 1)) : 1.0;
}

// OKS of person p against track t (t's pose is the ground truth)
HD double oks(const TrackSlot& t, const PersonPose& p, const double* var) {
    const unsigned both = t.mask & p.mask;
    if (!both) return 0.0;
    double s = 0.0;
    int m = 0;
    for (int j = 0; j < kCoco; j++) {
        if (!(both >> j & 1u)) continue;
        const long long dx = (long long) p.xy[2 * j] - t.xy[2 * j], dy = (long long) p.xy[2 * j + 1] - t.xy[2 * j + 1];
        const double e = (double) (dx * dx + dy * dy) / var[j] / t.area / 2.0;
        s += exp(-e);
        m++;
    }
    return s / m;
}

// the matching rule: the order of a person's candidate tracks (key: the track's tag, i.e. its id) and of a track's
// candidate people (key: the row) -- both the total order's restriction to pairs sharing that person or track.
// Liveness and the order in which the slots of unmatched live tracks are reused are common.cuh's expired / evict_first.
HD bool pair_first(double sa, int key_a, double sb, int key_b) { return sa > sb || (sa == sb && key_a < key_b); }

struct TrackArgs {
    const int* num_humans;   // [n]
    const ekp_peak* parts;   // [n][max_humans][18]
    int max_humans, F, max_tracks, max_age;
    double min_oks;
    double var[kCoco];       // oks_vars
    int* ids;                // [n][max_humans]
    unsigned char* state;    // [n_seq] x track_seq_bytes(max_tracks)
};

// one sequence's working set (shared memory on the device)
struct TrackWork {
    double* var;        // [17]
    TrackSlot* slot;    // [max_tracks]
    PersonPose* per;    // [max_humans]
    double* sim;        // [cache_cap] similarities of the frame, person-major over the live list
    int* live;          // [max_tracks] slots of the live tracks
    int* ltag;          // [max_tracks] their tags
    int* freel;         // [max_tracks] free slots, then the slots to reuse in reuse order
    int* tmatch;        // [max_tracks] per live track: matched person or -1
    int* tbest;         // [max_tracks] per live track: best free person of this round or -1
    int* pmatch;        // [max_humans] per person: matched live track or -1
    int* pbest;         // [max_humans] per person: best free live track of this round; then its birth rank
    int* cnt;           // [4] live, free, births
    int cache_cap;
};

// Carves the working set out of `base` (nullptr: only sizes it); returns its bytes.
HD size_t track_work_layout(int max_humans, int max_tracks, int cache_cap, unsigned char* base, TrackWork* w) {
    size_t off = 0;
    auto take = [&](size_t bytes) { unsigned char* p = base ? base + off : nullptr; off += (bytes + 15) & ~(size_t) 15; return p; };
    TrackWork t;
    t.var = (double*) take(sizeof(double) * kCoco);
    t.slot = (TrackSlot*) take(sizeof(TrackSlot) * max_tracks);
    t.per = (PersonPose*) take(sizeof(PersonPose) * max_humans);
    t.live = (int*) take(sizeof(int) * max_tracks);
    t.ltag = (int*) take(sizeof(int) * max_tracks);
    t.freel = (int*) take(sizeof(int) * max_tracks);
    t.tmatch = (int*) take(sizeof(int) * max_tracks);
    t.tbest = (int*) take(sizeof(int) * max_tracks);
    t.pmatch = (int*) take(sizeof(int) * max_humans);
    t.pbest = (int*) take(sizeof(int) * max_humans);
    t.cnt = (int*) take(sizeof(int) * 4);
    t.sim = (double*) take(sizeof(double) * cache_cap);
    t.cache_cap = cache_cap;
    if (w) *w = t;
    return off;
}

// sim[p * L + k] = OKS of person p against live track k, for the pairs of thread tid of nt.  Not inlined: the slow-path
// calls of the double divisions then save only this loop's registers, and the kernel needs no local memory.
__host__ __device__ __noinline__ void similarities(const TrackSlot* slot, const int* live, const PersonPose* per, const double* var,
                                                   double* sim, int P, int L, int tid, int nt) {
    for (int u = tid; u < P * L; u += nt) {
        const int p = u / L, k = u - p * L;
        sim[u] = oks(slot[live[k]], per[p], var);
    }
}

// The first of the lanes' candidates (best = -1: none), left in every lane; keys are unique within one choice, so the
// order is total and the result does not depend on the reduction order.  One lane (the host) has nothing to reduce.
HD void warp_first(int& best, double& bs, int& bkey, int lanes) {
#ifdef __CUDA_ARCH__
    for (int o = lanes / 2; o > 0; o >>= 1) {
        const int ob = __shfl_xor_sync(~0u, best, o), ok = __shfl_xor_sync(~0u, bkey, o);
        const double os = __shfl_xor_sync(~0u, bs, o);
        if (ob >= 0 && (best < 0 || pair_first(os, ok, bs, bkey))) { best = ob; bs = os; bkey = ok; }
    }
#endif
}

// Runs the F frames of sequence `seq` on thread `tid` of `nt`.
HD void track_sequence(const TrackArgs& A, int seq, const TrackWork& W, int tid, int nt) {
    const int MH = A.max_humans, MT = A.max_tracks;
    const int lanes = nt >= 32 ? 32 : 1, lane = tid % lanes, warp = tid / lanes, nwarps = nt / lanes;  // nt % 32 == 0 or nt == 1
    TrackHead* gh = reinterpret_cast<TrackHead*>(A.state + seq_bytes(MT) * (size_t) seq);
    const int* gs = reinterpret_cast<const int*>(gh + 1);
    double* gsim = reinterpret_cast<double*>(A.state + seq_bytes(MT) * (size_t) seq + slots_bytes(MT));
    const int words = (int) (sizeof(TrackSlot) / 4) * MT;
    for (int k = tid; k < words; k += nt) reinterpret_cast<int*>(W.slot)[k] = gs[k];
    for (int j = tid; j < kCoco; j += nt) W.var[j] = A.var[j];
    int f = gh->frame, next_id = gh->next_id;
    bar();
    for (int t = 0; t < A.F; t++, f++) {
        const int img = seq * A.F + t;
        const int P = min(max(A.num_humans[img], 0), MH);
        const ekp_peak* rows = A.parts + (size_t) img * MH * EKP_NUM_PART;
        int* ids = A.ids + (size_t) img * MH;
        if (tid == 0) W.cnt[0] = W.cnt[1] = W.cnt[2] = 0;
        bar();
        // 1. people, expiry, slot lists
        for (int p = tid; p < MH; p += nt) {
            if (p < P) { load_pose(rows + (size_t) p * EKP_NUM_PART, W.per[p]); W.pmatch[p] = -1; }
            else ids[p] = -1;
        }
        for (int k = tid; k < MT; k += nt) {
            TrackSlot& s = W.slot[k];
            if (s.tag && expired(s.last_seen, f, A.max_age)) s.tag = 0;
            if (s.tag) { const int q = claim(&W.cnt[0]); W.live[q] = k; W.ltag[q] = s.tag; }
            else W.freel[claim(&W.cnt[1])] = k;
        }
        bar();
        const int L = W.cnt[0], Fr = W.cnt[1];
        // 2. similarities: in shared memory when they fit, else in the sequence's scratch in the state
        double* sim = P * L <= W.cache_cap ? W.sim : gsim;
        similarities(W.slot, W.live, W.per, W.var, sim, P, L, tid, nt);
        for (int k = tid; k < L; k += nt) W.tmatch[k] = -1;
        bar();
        // 3. greedy matching by rounds of mutual first choices: one warp per free person or track finds its first choice
        if (P && L) {
            for (;;) {
                for (int u = warp; u < P + L; u += nwarps) {
                    int best = -1, bkey = 0;
                    double bs = 0.0;
                    if (u < P) {
                        if (W.pmatch[u] >= 0) continue;  // warp-uniform
                        for (int k = lane; k < L; k += lanes) {
                            if (W.tmatch[k] >= 0) continue;
                            const double s = sim[u * L + k];
                            if (s >= A.min_oks && (best < 0 || pair_first(s, W.ltag[k], bs, bkey))) { best = k; bs = s; bkey = W.ltag[k]; }
                        }
                        warp_first(best, bs, bkey, lanes);
                        if (lane == 0) W.pbest[u] = best;
                    } else {
                        const int k = u - P;
                        if (W.tmatch[k] >= 0) continue;
                        for (int p = lane; p < P; p += lanes) {
                            if (W.pmatch[p] >= 0) continue;
                            const double s = sim[p * L + k];
                            if (s >= A.min_oks && (best < 0 || pair_first(s, p, bs, bkey))) { best = p; bs = s; bkey = p; }
                        }
                        warp_first(best, bs, bkey, lanes);
                        if (lane == 0) W.tbest[k] = best;
                    }
                }
                bar();
                // a free person whose first choice was not mutual may still be matched in a later round; one whose
                // choice was none never will (tracks only get taken), so the rounds end when no such person is left
                int pending = 0;
                for (int p = tid; p < P; p += nt) {
                    if (W.pmatch[p] >= 0) continue;
                    const int k = W.pbest[p];
                    if (k >= 0 && W.tbest[k] == p) { W.pmatch[p] = k; W.tmatch[k] = p; }
                    else pending |= k >= 0;
                }
                if (!bar_or(pending)) break;
            }
        }
        // 4. matched tracks take their person's pose; the birth rank of every unmatched person
        for (int p = tid; p < P; p += nt) {
            const int k = W.pmatch[p];
            if (k >= 0) {
                TrackSlot& s = W.slot[W.live[k]];
                ids[p] = s.tag - 1;
                s.last_seen = f; s.mask = W.per[p].mask; s.area = W.per[p].area;
                for (int j = 0; j < 2 * kCoco; j++) s.xy[j] = W.per[p].xy[j];
            } else {
                int r = 0;
                for (int q = 0; q < p; q++) r += W.pmatch[q] < 0;
                W.pbest[p] = r;
                claim(&W.cnt[2]);
            }
        }
        bar();
        const int B = W.cnt[2];
        if (B > Fr) {  // every slot is taken: reuse those of the B - Fr oldest unmatched tracks
            for (int k = tid; k < L; k += nt) {
                const TrackSlot& s = W.slot[W.live[k]];
                if (s.last_seen == f) continue;  // matched in this frame
                int r = 0;
                for (int q = 0; q < L; q++) {
                    const TrackSlot& o = W.slot[W.live[q]];
                    r += o.last_seen != f && evict_first(o.last_seen, o.tag, s.last_seen, s.tag);  // tags order as ids
                }
                if (r < B - Fr) W.freel[Fr + r] = W.live[k];
            }
            bar();
        }
        for (int p = tid; p < P; p += nt) {
            if (W.pmatch[p] >= 0) continue;
            const int r = W.pbest[p];
            TrackSlot& s = W.slot[W.freel[r]];
            s.tag = next_id + r + 1;
            s.last_seen = f; s.mask = W.per[p].mask; s.area = W.per[p].area;
            for (int j = 0; j < 2 * kCoco; j++) s.xy[j] = W.per[p].xy[j];
            ids[p] = next_id + r;
        }
        next_id += B;
        bar();
    }
    int* gw = reinterpret_cast<int*>(gh + 1);
    for (int k = tid; k < words; k += nt) gw[k] = reinterpret_cast<const int*>(W.slot)[k];
    if (tid == 0) { gh->frame = f; gh->next_id = next_id; }
}

__global__ void __launch_bounds__(kTrackThreads) track_kernel(const TrackArgs A, int cache_cap) {
    extern __shared__ __align__(16) unsigned char smem[];
    TrackWork W;
    track_work_layout(A.max_humans, A.max_tracks, cache_cap, smem, &W);
    track_sequence(A, blockIdx.x, W, threadIdx.x, blockDim.x);
}

cudaError_t configure_track() {
    return cudaFuncSetAttribute(track_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) kTrackSmemMax);
}

// the shared similarity matrix takes what the rest of the working set leaves of the block's shared memory, up to P x L pairs
// (at max_humans = max_tracks = EKP_LIMIT_TRACKS the rest takes 174,240 of the 232,448 bytes: 7,276 similarities)
static int track_cache_cap(int max_humans, int max_tracks) {
    const size_t rest = track_work_layout(max_humans, max_tracks, 0, nullptr, nullptr);
    const size_t room = (kTrackSmemMax - rest) / sizeof(double);
    return (int) (room < (size_t) max_humans * max_tracks ? room : (size_t) max_humans * max_tracks);
}

cudaError_t launch_track(const int* num_humans, const ekp_peak* parts, int n, int max_humans, void* state, int n_seq, int max_tracks,
                         float min_oks, int max_age, int* ids, cudaStream_t stream) {
    TrackArgs A = {num_humans, parts, max_humans, n / n_seq, max_tracks, max_age, (double) min_oks, {}, ids,
                   static_cast<unsigned char*>(state)};
    oks_vars(A.var);
    const int cap = track_cache_cap(max_humans, max_tracks);
    const size_t smem = track_work_layout(max_humans, max_tracks, cap, nullptr, nullptr);
    track_kernel<<<n_seq, kTrackThreads, smem, stream>>>(A, cap);
    return cudaGetLastError();
}

void debug_track_host(const int* num_humans, const ekp_peak* parts, int n, int max_humans, void* state, int n_seq, int max_tracks,
                      float min_oks, int max_age, int* ids) {
    TrackArgs A = {num_humans, parts, max_humans, n / n_seq, max_tracks, max_age, (double) min_oks, {}, ids,
                   static_cast<unsigned char*>(state)};
    oks_vars(A.var);
    const int cap = track_cache_cap(max_humans, max_tracks);  // as on the device: the same frames use the state's scratch
    std::vector<double> buf(track_work_layout(max_humans, max_tracks, cap, nullptr, nullptr) / sizeof(double) + 2);
    TrackWork W;
    track_work_layout(max_humans, max_tracks, cap, reinterpret_cast<unsigned char*>(buf.data()), &W);
    for (int s = 0; s < n_seq; s++) track_sequence(A, s, W, 0, 1);
}

}  // namespace ekp
