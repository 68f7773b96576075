// process_paf.cu -- the reference's process_paf / get_* operator surface (lib/pafprocess/pafprocess.h:53-59) on the
// library's kernels: stages 4-5 for peaks and a paf_mat in host memory, run on a context of its own, with the results
// kept process-global like the reference's.
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <mutex>
#include <vector>

#include "capi.cuh"

using namespace ekp;

namespace {
// pafprocess.h:16-24 on the host: the two parts of each limb, and the x channel of its PAF (y = x + 1)
const int kHostPairs[EKP_NUM_LIMB][2] = {{1, 2}, {1, 5}, {2, 3}, {3, 4}, {5, 6}, {6, 7}, {1, 8}, {8, 9}, {9, 10}, {1, 11},
                                         {11, 12}, {12, 13}, {1, 0}, {0, 14}, {14, 16}, {0, 15}, {15, 17}, {2, 16}, {5, 17}};
const int kHostPairsNet[EKP_NUM_LIMB] = {12, 20, 14, 16, 22, 24, 0, 2, 4, 6, 8, 10, 28, 30, 34, 32, 36, 18, 26};

// Process-global "last result", like the reference's globals (pafprocess.cpp:12-13).
std::mutex g_mu;   // guards everything of this file
ekp_ctx* g_ctx = nullptr;
std::vector<float> g_subset;      // [num_humans][20]
std::vector<float> g_hscore;      // [num_humans] subset[18] / subset[19], computed on the device
std::vector<ekp_peak> g_line;     // part-sorted peak table
int g_num_humans = 0;

// the listed route: one block [pair prefix | peaks | samples], pinned on the host and (copying form) on the device
const long long kListedMaxSamples = 64 * 1024;
unsigned char* g_listed_host = nullptr; size_t g_listed_host_cap = 0;
unsigned char* g_listed_dev = nullptr; size_t g_listed_dev_cap = 0;
unsigned char* g_listed_host_dev = nullptr;   // the device's view of g_listed_host
const int kSmallPeaks = 512;
const long long kSmallMaxSamples = 16384;

// the uploaded route: the peaks, and the sample offsets (device + pinned host), gathered samples (pinned host + device) and
// pair prefix of the sparse upload, or the whole paf_mat
float* g_dev_peaks = nullptr; size_t g_dev_peaks_cap = 0;
unsigned* g_dev_offs = nullptr; size_t g_dev_offs_cap = 0;
unsigned* g_host_offs = nullptr; size_t g_host_offs_cap = 0;
float2* g_host_samp = nullptr; size_t g_host_samp_cap = 0;
float2* g_dev_samp = nullptr; size_t g_dev_samp_cap = 0;
int* g_dev_pair_base = nullptr;
float* g_dev_paf = nullptr; size_t g_dev_paf_cap = 0;
const long long kSparseMaxSamples = 8ll << 20;  // beyond this the whole tensor is uploaded instead

// capacities of the context a scene needs, grown by grow_for
struct Need { int humans = 128, part = EKP_MAX_PART, cand = EKP_MAX_CAND; };

// The context behind the operator surface: re-created with larger capacities when a scene needs them (the new one
// first, so a failed creation leaves the old one in place), never beyond the library's limits.  Its graphs go with it.
int compat_ctx(long long npk, const Need& need) {
    if (g_ctx && g_ctx->max_peaks >= npk && g_ctx->max_humans >= need.humans && g_ctx->max_part >= need.part &&
        g_ctx->max_cand >= need.cand)
        return EKP_OK;
    int dev = 0;
    if (const char* s = getenv("EKP_DEVICE")) dev = atoi(s);
    int peaks = 1024, humans = 128;
    while (peaks < npk) peaks *= 2;
    while (humans < need.humans) humans *= 2;
    peaks = std::min(peaks, EKP_LIMIT_PEAKS);
    humans = std::min(humans, EKP_LIMIT_HUMANS);
    int part = need.part, cand = need.cand;
    if (g_ctx) { part = std::max(part, g_ctx->max_part); cand = std::max(cand, g_ctx->max_cand); }
    ekp_ctx* fresh = nullptr;
    int rc = ekp_create_ex(&fresh, dev, 1, 8, 8, peaks, humans, std::min(part, EKP_LIMIT_PART), std::min(cand, EKP_LIMIT_CAND));
    if (rc) return rc;
    if (g_ctx) ekp_destroy(g_ctx);
    g_ctx = fresh;
    return EKP_OK;
}

// The prefix over the limbs of their candidate pairs, stage 4's sample layout, for count[part] peaks of each part of
// which at most max_part take part: pair_base[0 .. EKP_NUM_LIMB].  Returns the number of pairs.
long long pair_prefix(const int* count, int max_part, int* pair_base) {
    long long acc = 0;
    for (int l = 0; l < EKP_NUM_LIMB; l++) {
        pair_base[l] = (int) acc;
        acc += (long long) std::min(count[kHostPairs[l][0]], max_part) * std::min(count[kHostPairs[l][1]], max_part);
    }
    pair_base[EKP_NUM_LIMB] = (int) acc;
    return acc;
}

// The part-sorted peak table of stage 4 from `npk` peak rows on the device, by the general ingest and sort kernels
// (a peak's id is its row).
int ingest_and_sort(ekp_ctx* c, const float* dev_peaks, int npk, int p3, int f1, int f2, cudaStream_t st) {
    CU(cudaMemsetAsync(c->raw_count, 0, sizeof(int) * 2 * (size_t) c->max_batch, st));
    CU(launch_peaks_ingest(dev_peaks, nullptr, npk, npk, p3, 1, f2, f1, c->raw, c->raw_count, c->max_peaks, c->overflow, st));
    c->launches += 1;
    return run_peak_sort(c, 1, /*id_from_key=*/1, st);
}

// After a capacity overflow: grows exactly what overflowed, within the library's limits, and says whether to run again.
// Too many peaks, an invalid peak, or a capacity already at its limit: the error stands.
bool grow_for(unsigned ovf, const ekp_ctx* c, Need& need) {
    if (ovf & (EKP_OVF_PEAKS | EKP_OVF_BADPEAK)) return false;
    bool grew = false, stuck = false;
    auto step = [&](unsigned bit, int have, int limit, int& want) {
        if (!(ovf & bit)) return;
        if (have < limit) { want = std::min(have * 4, limit); grew = true; }
        else stuck = true;
    };
    step(EKP_OVF_HUMANS, c->max_humans, EKP_LIMIT_HUMANS, need.humans);
    step(EKP_OVF_PART, c->max_part, EKP_LIMIT_PART, need.part);
    step(EKP_OVF_CANDIDATES, c->max_cand, EKP_LIMIT_CAND, need.cand);
    return grew && !stuck;
}

// ---- the listed route: everything stage 4 needs in ONE upload, no mid-call synchronisation --------------------------
// For up to kListedMaxSamples samples the host lists them itself: it buckets the caller's peaks by part (the order of
// the reference's own buckets, pafprocess.cpp:24-43), walks the pairs of every limb in the kernel's order (a outer,
// b inner) and copies the two floats at each of the <= 10 sample positions out of the caller's paf_mat -- the positions
// by the roundpaf arithmetic of pafprocess.cpp:228-233, 240-242, which is index arithmetic on the INPUT, not scoring:
// unit vectors, dot products, both criteria, sort, assignment and assembly all run in the kernels, on these values.
// One pinned block [pair prefix | peaks | samples] -> one H2D copy -> ingest, sort, connect (PAF_PACKED), assemble ->
// one D2H copy of the result record -> one wait.  The part-sorted peak table the getters index (pafprocess.cpp:208-218)
// is the bucket order itself, so it never has to come back from the device: it is returned in `line`.
// Returns 1 when the scene is not eligible (an invalid peak, a part over max_part, too many samples): the uploaded
// route then runs and reports whatever is wrong.
int process_paf_listed(ekp_ctx* c, long long npk, int p3, const float* peaks, int h1, int f1, int f2, int f3, const float* pafmap,
                       std::vector<ekp_peak>& line) {
    std::vector<int> bucket[EKP_NUM_PART];
    for (long long k = 0; k < npk; k++) {
        const float* row = peaks + k * p3;
        const float pt = row[4];
        const int part = pt > -1.f && pt < (float) EKP_NUM_PART ? (int) pt : -1;
        const int x = (int) row[0], y = (int) row[1];   // C truncation, pafprocess.cpp:30-31
        if (part < 0 || !(row[0] > -1.f && row[0] < (float) f2 + 1.f) || !(row[1] > -1.f && row[1] < (float) f1 + 1.f) || x < 0 || x >= f2 ||
            y < 0 || y >= f1 || !(row[2] == row[2]))
            return 1;
        bucket[part].push_back((int) k);
    }
    int count[EKP_NUM_PART];
    for (int part = 0; part < EKP_NUM_PART; part++) {
        count[part] = (int) bucket[part].size();
        if (count[part] > c->max_part) return 1;
    }
    int pair_base[32] = {0};
    const long long nsamples = pair_prefix(count, c->max_part, pair_base) * 10;
    if (nsamples > kListedMaxSamples) return 1;
    // Small scenes (a handful of people: every frame of an ordinary video).  Such a call used to wait ~25 us for the device-side
    // chain H2D copy -> 3 kernels -> D2H copy -> event after spending ~25 us submitting it (70 us at 3 people).  Here the
    // kernels read the pinned block and write the result record THROUGH PCIe themselves (zero-copy: a few KB, one round trip
    // per kernel), so the chain is the three kernels; and the block has a fixed layout (room for kSmallPeaks peaks, samples
    // rounded up to a size class, the peak count inside), so the launch arguments depend only on (shape, size class) and the
    // three launches are replayed as ONE CUDA graph launch (1.5 us to submit).  Measured, raw call at 3 / 8 people: 70 / 112 us
    // before, 58 / 111 us zero-copy with eager launches (what EKP_GRAPHS=0 runs), 51 / 103 us as a graph (the copies inside a
    // graph instead: 66 / 116 us; profiles/README.md).  What is left is the latency of the three kernels themselves (~35 us).
    const bool small = c->h_records_dev && npk <= kSmallPeaks && npk <= peaks_one_max() && nsamples <= kSmallMaxSamples;
    long long samp_class = 2048;
    while (samp_class < nsamples) samp_class *= 2;
    pair_base[31] = (int) npk;
    const size_t off_peaks = sizeof(pair_base);
    const size_t off_samp = (off_peaks + sizeof(float) * (size_t) (small ? kSmallPeaks : npk) * p3 + 7) & ~(size_t) 7;
    const size_t bytes = off_samp + sizeof(float2) * (size_t) (small ? samp_class : (nsamples > 0 ? nsamples : 1));
    if (g_listed_host_cap < bytes || g_listed_dev_cap < bytes) {
        drop_graphs(c);   // they read the old block
        int rc = grow(g_listed_host, g_listed_host_cap, bytes, GROW_PINNED | GROW_SLACK);
        if (rc == EKP_OK) rc = grow(g_listed_dev, g_listed_dev_cap, bytes, GROW_SLACK);
        if (rc) return rc;
        if (cudaHostGetDevicePointer((void**) &g_listed_host_dev, g_listed_host, 0) != cudaSuccess) { cudaGetLastError(); g_listed_host_dev = nullptr; }
    }
    memcpy(g_listed_host, pair_base, sizeof(pair_base));
    memcpy(g_listed_host + off_peaks, peaks, sizeof(float) * (size_t) npk * p3);
    float2* samp = reinterpret_cast<float2*>(g_listed_host + off_samp);
    size_t k = 0;
    for (int l = 0; l < EKP_NUM_LIMB; l++) {
        const std::vector<int>& A = bucket[kHostPairs[l][0]];
        const std::vector<int>& B = bucket[kHostPairs[l][1]];
        const float* chan = pafmap + kHostPairsNet[l];
        for (int ia : A) {
            const int ax = (int) peaks[(size_t) ia * p3], ay = (int) peaks[(size_t) ia * p3 + 1];
            for (int ib : B) {
                const int bx = (int) peaks[(size_t) ib * p3], by = (int) peaks[(size_t) ib * p3 + 1];
                volatile float step_x = (float) (bx - ax) / 10.0f, step_y = (float) (by - ay) / 10.0f;   // pafprocess.cpp:224-225
                for (int i = 0; i < 10; i++) {
                    volatile float fx = (float) i * step_x, fy = (float) i * step_y;   // float products, then float sums (:228),
                    volatile float sx = (float) ax + fx, sy = (float) ay + fy;         // rounded one by one like the C++ (no contraction)
                    int lx = (int) ((double) sx + 0.5), ly = (int) ((double) sy + 0.5);  // roundpaf, :240-242
                    lx = std::min(std::max(lx, 0), f2 - 1);
                    ly = std::min(std::max(ly, 0), f1 - 1);
                    const float* q = chan + ((size_t) ly * f2 + lx) * f3;
                    samp[k++] = make_float2(q[0], q[1]);
                }
            }
        }
    }
    line.clear();
    line.reserve((size_t) npk);
    for (int part = 0; part < EKP_NUM_PART; part++)   // peak_infos_line: the buckets one after the other (pafprocess.cpp:38-43)
        for (int kk : bucket[part]) {
            const float* row = peaks + (size_t) kk * p3;
            ekp_peak pk;
            pk.x = (int) row[0]; pk.y = (int) row[1]; pk.score = row[2]; pk.id = kk;
            line.push_back(pk);
        }
    // Small scenes: the kernels read the pinned block itself and write the record into pinned memory.  Otherwise the block
    // is copied to the device first and the record comes back with the packed D2H copy.
    const bool zero_copy = small && g_listed_host_dev;
    const unsigned char* blk = zero_copy ? g_listed_host_dev : g_listed_dev;
    const PafSource src = paf_source(PAF_PACKED, blk + off_samp, reinterpret_cast<const int*>(blk), f1, f2, f3);
    auto enqueue = [&](cudaStream_t q) -> int {
        const float* blk_peaks = reinterpret_cast<const float*>(blk + off_peaks);
        if (npk <= peaks_one_max()) {   // ingest + sort in one block, no counters to clear; the peak count is in the block
            CU(launch_peaks_ingest_sort_one(blk_peaks, 0, reinterpret_cast<const int*>(blk) + 31, p3, f2, f1, c->max_peaks, c->max_part, c->line,
                                            c->part_off, c->n_peaks, c->raw_count, c->overflow, q));
            c->launches += 1;
        } else {
            int rc = ingest_and_sort(c, blk_peaks, (int) npk, p3, f1, f2, q);
            if (rc) return rc;
        }
        return run_connect_assemble(c, 1, src, h1, q, /*host_copy=*/true, zero_copy ? c->h_records_dev : nullptr);
    };
    const cudaStream_t st = nullptr;
    if (zero_copy) return launch_cached(c, GraphKey{{}, {p3, f1, f2, f3, h1, (long long) bytes}}, 0, st, enqueue);
    CU(cudaMemcpyAsync(g_listed_dev, g_listed_host, bytes, cudaMemcpyHostToDevice, st));
    return enqueue(st);
}

// ---- the uploaded route: the peaks go up as they are and the device sorts them -------------------------------------
// Sparse upload: stage 4 reads at most 10 positions of paf_mat per candidate pair, a few KB against the 24 MB tensor.
// Pairs per limb follow from the part column of the caller's peaks; a kernel lists the positions, the host gathers the
// values.  Otherwise (or beyond kSparseMaxSamples samples) the whole tensor is uploaded.
int process_paf_uploaded(ekp_ctx* c, long long npk, int p3, const float* peaks, int h1, int f1, int f2, int f3, const float* pafmap,
                         bool sparse) {
    const size_t pk_elems = (size_t) npk * p3, paf_elems = (size_t) f1 * f2 * f3;
    int rc = grow(g_dev_peaks, g_dev_peaks_cap, pk_elems);
    if (rc) return rc;
    int pair_base[EKP_NUM_LIMB + 1];
    long long nsamples = 0;
    if (sparse) {
        int per_part[EKP_NUM_PART] = {0};
        for (long long k = 0; k < npk; k++) {
            const float pt = peaks[k * p3 + 4];
            const int part = pt > -1.f && pt < (float) EKP_NUM_PART ? (int) pt : -1;  // (int) truncates like the ingest kernel;
            if (part >= 0) per_part[part]++;  // any peak it rejects for another reason fails the whole call (EKP_OVF_BADPEAK)
        }
        nsamples = pair_prefix(per_part, c->max_part, pair_base) * 10;
        sparse = nsamples <= kSparseMaxSamples;
    }
    const cudaStream_t st = nullptr;
    CU(cudaMemcpyAsync(g_dev_peaks, peaks, pk_elems * sizeof(float), cudaMemcpyHostToDevice, st));
    rc = ingest_and_sort(c, g_dev_peaks, (int) npk, p3, f1, f2, st);
    if (rc) return rc;
    if (sparse && nsamples > 0) {
        const size_t ns = (size_t) nsamples;
        rc = grow(g_dev_offs, g_dev_offs_cap, ns, GROW_SLACK);
        if (rc == EKP_OK) rc = grow(g_dev_samp, g_dev_samp_cap, ns, GROW_SLACK);
        if (rc == EKP_OK) rc = grow(g_host_offs, g_host_offs_cap, ns, GROW_PINNED | GROW_SLACK);
        if (rc == EKP_OK) rc = grow(g_host_samp, g_host_samp_cap, ns, GROW_PINNED | GROW_SLACK);
        if (rc) return rc;
        if (!g_dev_pair_base) CU(cudaMalloc((void**) &g_dev_pair_base, sizeof(int) * (EKP_NUM_LIMB + 1)));
        CU(cudaMemcpyAsync(g_dev_pair_base, pair_base, sizeof(pair_base), cudaMemcpyHostToDevice, st));
        CU(cudaMemsetAsync(g_dev_offs, 0, ns * sizeof(unsigned), st));  // limbs the kernel skips stay in bounds
        CU(launch_pair_sample_offsets(c->line, c->part_off, g_dev_pair_base, f1, f2, f3, c->max_part, g_dev_offs, st));
        c->launches += 1;
        CU(cudaMemcpyAsync(g_host_offs, g_dev_offs, ns * sizeof(unsigned), cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        for (size_t k = 0; k < ns; k++) {  // the gather: a copy, no arithmetic
            const float* q = pafmap + g_host_offs[k];
            g_host_samp[k] = make_float2(q[0], q[1]);
        }
        CU(cudaMemcpyAsync(g_dev_samp, g_host_samp, ns * sizeof(float2), cudaMemcpyHostToDevice, st));
        return run_connect_assemble(c, 1, paf_source(PAF_PACKED, g_dev_samp, g_dev_pair_base, f1, f2, f3), h1, st, /*host_copy=*/true);
    }
    rc = grow(g_dev_paf, g_dev_paf_cap, paf_elems);
    if (rc) return rc;
    CU(cudaMemcpyAsync(g_dev_paf, pafmap, paf_elems * sizeof(float), cudaMemcpyHostToDevice, st));
    return run_connect_assemble(c, 1, paf_source(PAF_FULL_HWC, g_dev_paf, nullptr, f1, f2, f3), h1, st, /*host_copy=*/true);
}

// the getters' view of a finished run
void publish(const ekp_ctx* c, int nh, const std::vector<float>& subset, std::vector<ekp_peak>& line) {
    g_num_humans = nh;
    g_subset.assign(subset.begin(), subset.begin() + (size_t) nh * 20);
    const float* hs = reinterpret_cast<const float*>(c->h_records + c->lay.off_hscore);
    g_hscore.assign(hs, hs + nh);
    g_line.swap(line);
}
}  // namespace

// Everything runs on the legacy default stream, and every call waits for its results.
extern "C" int process_paf(int p1, int p2, int p3, float* peaks, int h1, int h2, int h3, float* heatmap, int f1, int f2,
                           int f3, float* pafmap) {
    (void) h2; (void) h3; (void) heatmap;  // heat_mat is used only through h1 (pafprocess.cpp:83)
    std::lock_guard<std::mutex> lock(g_mu);
    g_num_humans = 0; g_subset.clear(); g_hscore.clear(); g_line.clear();
    if (p1 < 0 || p2 < 0 || p3 < 5 || f1 < 1 || f2 < 1 || f3 < 38 || !pafmap || (!peaks && (long long) p1 * p2 > 0))
        return fail(EKP_ERR_ARG, "process_paf: bad arguments (peaks [%d,%d,%d] needs p3 >= 5, paf [%d,%d,%d] needs f3 >= 38)", p1, p2, p3, f1, f2, f3);
    const long long npk = (long long) p1 * p2;  // all p1 "images" are pooled (pafprocess.cpp:26-36)
    if (npk > EKP_LIMIT_PEAKS) return fail(EKP_ERR_CAPACITY, "process_paf: %lld peaks > %d", npk, EKP_LIMIT_PEAKS);
    if (npk == 0) return EKP_OK;  // nothing to connect: zero humans, like the reference
    const bool offsets_fit = (size_t) f1 * f2 * f3 < (1ull << 32);   // sample positions are 32-bit offsets into paf_mat
    Need need;
    for (int attempt = 0; attempt < 8; attempt++) {
        int rc = compat_ctx(npk, need);
        if (rc) return rc;
        ekp_ctx* c = g_ctx;
        CU(cudaSetDevice(c->device));
        // EKP_PROCESS_PAF_UPLOAD = listed (default) | sparse | dense forces a route; read on every call
        const char* route = getenv("EKP_PROCESS_PAF_UPLOAD");
        std::vector<ekp_peak> line;
        rc = offsets_fit && (!route || strcmp(route, "listed") == 0) ? process_paf_listed(c, npk, p3, peaks, h1, f1, f2, f3, pafmap, line) : 1;
        const bool listed = rc == EKP_OK;
        if (rc == 1) rc = process_paf_uploaded(c, npk, p3, peaks, h1, f1, f2, f3, pafmap, offsets_fit && !(route && strcmp(route, "dense") == 0));
        if (rc == EKP_OK) rc = finish_submit(c, 1, nullptr, /*records_on_host=*/true);
        if (rc) return rc;
        std::vector<float> subset((size_t) c->max_humans * 20);
        int nh = 0, np = 0;
        unsigned ovf = 0;
        if (!listed) line.resize((size_t) c->max_peaks);   // the device's part-sorted table
        rc = ekp_results(c, &nh, subset.data(), &np, listed ? nullptr : line.data(), &ovf);
        if (rc == EKP_ERR_CAPACITY && grow_for(ovf, c, need)) continue;
        if (rc) return rc;
        if (!listed) line.resize((size_t) np);
        publish(c, nh, subset, line);
        return EKP_OK;  // the reference returns 0 (pafprocess.cpp:193)
    }
    return fail(EKP_ERR_CAPACITY, "process_paf: the scene does not fit the library's limits");
}

extern "C" int get_num_humans(void) { return g_num_humans; }
extern "C" int get_part_cid(int human_id, int part_id) {
    if (human_id < 0 || human_id >= g_num_humans || part_id < 0 || part_id >= EKP_SUBSET_COLS) { fail(EKP_ERR_ARG, "get_part_cid(%d, %d) out of range", human_id, part_id); return -1; }
    return (int) g_subset[(size_t) human_id * 20 + part_id];
}
extern "C" float get_score(int human_id) {
    if (human_id < 0 || human_id >= g_num_humans) { fail(EKP_ERR_ARG, "get_score(%d) out of range", human_id); return 0.f; }
    return g_hscore[(size_t) human_id];
}
static const ekp_peak* peak_at(int cid, const char* who) {
    if (cid < 0 || (size_t) cid >= g_line.size()) { fail(EKP_ERR_ARG, "%s(%d) out of range", who, cid); return nullptr; }
    return &g_line[(size_t) cid];
}
extern "C" int get_part_x(int cid) { const ekp_peak* p = peak_at(cid, "get_part_x"); return p ? p->x : 0; }
extern "C" int get_part_y(int cid) { const ekp_peak* p = peak_at(cid, "get_part_y"); return p ? p->y : 0; }
extern "C" float get_part_score(int cid) { const ekp_peak* p = peak_at(cid, "get_part_score"); return p ? p->score : 0.f; }
