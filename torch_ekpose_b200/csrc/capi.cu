// capi.cu -- the C ABI of libekpose_b200.so (include/ekpose_b200.h): context and work buffers,
// the batched device API, and the reference's process_paf / get_* operator surface
// (/root/reference/lib/pafprocess/pafprocess.h:53-59) on top of the same kernels.
// Host code only orchestrates: every stage of the path runs in the CUDA kernels of this
// directory and there is no CPU implementation to fall back to.
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include <algorithm>
#include <atomic>
#include <mutex>
#include <vector>

#include "common.cuh"

namespace ekp {
// kernels (one translation unit each)
size_t dense_frontend_smem_bytes(int tile_wl, bool materialise);
int dense_frontend_tile_wl(int w);
cudaError_t configure_dense_frontend();
cudaError_t configure_dense_plane(int max_h, int max_w);
cudaError_t set_interior_taps(const float* taps64);
cudaError_t set_cubic_table(const float* tab32);
cudaError_t launch_dense_frontend(const DenseParams& p, cudaStream_t stream);
cudaError_t launch_ref_frontend(const RefParams& p, cudaStream_t stream);
int ref_frontend_launches(int refine);
cudaError_t configure_ref_frontend(int max_h, int max_w);
cudaError_t launch_upsample_nearest(const float* lo, int layout, int n, int h, int w, int C, float* out, cudaStream_t stream);
cudaError_t launch_peaks_ingest(const float* peaks, const int* n_peaks, int n_fixed, int peaks_stride, int p3, int n, int W,
                                int H, RawPeak* raw, int* raw_count, int raw_cap, unsigned* overflow, cudaStream_t stream);
cudaError_t configure_peaks_sort(int raw_cap);
int peaks_one_max();
cudaError_t launch_peaks_ingest_sort_one(const float* peaks, int npk, const int* npk_dev, int p3, int W, int H, int raw_cap, int max_part,
                                         ekp_peak* line, int* part_off, int* n_peaks, int* raw_count, unsigned* overflow, cudaStream_t stream);
cudaError_t launch_peaks_sort(const RawPeak* raw, const int* raw_count, int raw_cap, int max_part, int id_from_key, int n,
                              ekp_peak* line, int* part_off, int* n_peaks, unsigned* overflow, cudaStream_t stream);
cudaError_t configure_connect(int max_part, int max_cand);
cudaError_t launch_paf_connect(const ConnectParams& P, int n, cudaStream_t stream);
cudaError_t configure_assemble(int max_humans, int max_peaks, int max_part);
cudaError_t launch_assemble(AsmParams P, int n, cudaStream_t stream);
cudaError_t launch_pair_sample_offsets(const ekp_peak* line, const int* part_off, const int* pair_base, int H, int W, int C,
                                       int max_part, unsigned* offs, cudaStream_t stream);
size_t debug_std_sort_scratch_words(int n);
cudaError_t launch_debug_std_sort(float* scores, unsigned* tags, int n, unsigned* scratch, cudaStream_t stream);
cudaError_t launch_preprocess(const unsigned char* src, float* out, const int* xofs, const short* ialpha, const int* yofs,
                              const short* ibeta, int n, int sh, int sw, int rh, int rw, int ph, int pw, int mode,
                              cudaStream_t stream);
cudaError_t launch_widen(const void* heat16, const void* paf16, size_t n_heat, size_t n_paf, int dtype, float* heat, float* paf,
                         cudaStream_t stream);
cudaError_t launch_draw(const unsigned char* records, const ResultLayout& lay, int max_humans, int map_h, int map_w,
                        unsigned char* frames, int n, int H, int W, unsigned* keys, unsigned epoch, cudaStream_t stream);
void debug_raster_host(int kind, int x0, int y0, int x1, int y1, int H, int W, unsigned char* mask);
void debug_draw_host(const int* num_humans, const ekp_peak* parts, int max_humans, int map_h, int map_w,
                     unsigned char* frames, int n, int H, int W);
}  // namespace ekp

using namespace ekp;

// ---- error reporting -------------------------------------------------------------------------
static thread_local char g_err[512] = "";
static int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}
#define CU(expr)                                                                                        \
    do {                                                                                                \
        cudaError_t _e = (expr);                                                                        \
        if (_e != cudaSuccess) return fail(EKP_ERR_CUDA, "%s: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)

extern "C" const char* ekp_last_error(void) { return g_err; }
extern "C" const char* ekp_version(void) { return "ekpose_b200 0.1 (sm_100a)"; }

// ---- host-side tables --------------------------------------------------------------------------
// Composite operator  A = Gaussian(sigma 3, radius 12, scipy 'reflect')  x  bilinear x8 (half-pixel,
// clamp) for an axis with n stride-8 samples, as 5 taps on stride-8 samples starting at
// clamp(D/8 - 2, 0, n-5).  Built in double and rounded once, in the accumulation order the
// oracle defines (oracle/frontend_oracle.c okp_dense_tables), padded to 8 floats per row.
static int reflect_idx(int i, int n) {
    while (i < 0 || i >= n) { if (i < 0) i = -i - 1; if (i >= n) i = 2 * n - 1 - i; }
    return i;
}
static int build_dense_taps(int n, std::vector<float>& taps) {
    const int N = 8 * n;
    if (n < 5) return -1;
    double wd[25], sum = 0.0;
    for (int j = -12; j <= 12; j++) { wd[j + 12] = exp(-0.5 * (double) (j * j) / 9.0); sum += wd[j + 12]; }
    for (int j = 0; j < 25; j++) wd[j] /= sum;
    taps.assign((size_t) N * 8, 0.f);
    std::vector<double> row(n);
    for (int D = 0; D < N; D++) {
        for (int i = 0; i < n; i++) row[i] = 0.0;
        for (int j = -12; j <= 12; j++) {
            const int Dp = reflect_idx(D + j, N);
            int i0 = (Dp + 4) / 8 - 1;
            const double t = (double) (2 * ((Dp + 4) % 8) + 1) / 16.0;
            const int i1 = i0 + 1 > n - 1 ? n - 1 : i0 + 1;
            if (i0 < 0) i0 = 0;
            row[i0] += wd[j + 12] * (1.0 - t);
            row[i1] += wd[j + 12] * t;
        }
        int base = D / 8 - 2;
        if (base < 0) base = 0;
        if (base > n - 5) base = n - 5;
        for (int i = 0; i < n; i++)
            if (row[i] != 0.0 && (i < base || i >= base + 5)) return -2;  // support must fit the window
        double tsum = 0.0;
        for (int k = 0; k < 5; k++) {
            taps[(size_t) D * 8 + k] = (float) row[base + k];
            if (row[base + k] < 0.0) return -3;
            tsum += (double) taps[(size_t) D * 8 + k];
        }
        if (tsum > 1.0 + 1e-6) return -3;  // the kernel's early-out relies on convex weights
    }
    return 0;
}
// cv2 interpolateCubic (A = -0.75) in float arithmetic for t = (2k+1)/16; volatile keeps the host
// compiler from contracting or reassociating.
static void build_cubic_table(float* tab /* [8][4] */) {
    for (int k = 0; k < 8; k++) {
        volatile float x = (float) (2 * k + 1) / 16.0f;
        const float A = -0.75f;
        volatile float x1 = x + 1, xm = 1 - x;
        volatile float c0 = A * x1; c0 = c0 - 5 * A; c0 = c0 * x1; c0 = c0 + 8 * A; c0 = c0 * x1; c0 = c0 - 4 * A;
        volatile float c1 = (A + 2) * x; c1 = c1 - (A + 3); c1 = c1 * x; c1 = c1 * x; c1 = c1 + 1;
        volatile float c2 = (A + 2) * xm; c2 = c2 - (A + 3); c2 = c2 * xm; c2 = c2 * xm; c2 = c2 + 1;
        volatile float c3 = 1.f - c0; c3 = c3 - c1; c3 = c3 - c2;
        tab[k * 4 + 0] = c0; tab[k * 4 + 1] = c1; tab[k * 4 + 2] = c2; tab[k * 4 + 3] = c3;
    }
}

// scipy.ndimage's Gaussian kernel for sigma = 3 (radius int(4 * 3 + 0.5) = 12), the 13 distinct weights w[-12] .. w[0]:
// _gaussian_kernel1d computes exp(-0.5 / sigma^2 * x^2) / sum in double, the sum being numpy's pairwise add.reduce of 25
// doubles (8 running sums over the first 24, ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)), then the 25th).  tests/test_oracle_pinning.py
// compares oracle/frontend_oracle.c's copy of this with scipy's own array, tests/test_abi.py this one with the oracle's.
static void build_scipy_gauss3(double* fw /* [13] */) {
    volatile double phi[25], r[8];
    for (int j = -12; j <= 12; j++) phi[j + 12] = exp(-0.5 / 9.0 * (double) (j * j));
    for (int j = 0; j < 8; j++) r[j] = phi[j];
    for (int i = 8; i < 24; i += 8)
        for (int j = 0; j < 8; j++) r[j] = r[j] + phi[i + j];
    volatile double sum = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
    sum = sum + phi[24];
    for (int j = 0; j < 13; j++) fw[j] = phi[j] / sum;
}
extern "C" int ekp_scipy_gauss3_weights(double* out13) {
    if (!out13) return fail(EKP_ERR_ARG, "ekp_scipy_gauss3_weights: NULL");
    build_scipy_gauss3(out13);
    return EKP_OK;
}

// ---- context -----------------------------------------------------------------------------------
// arguments of one batch submission (also the key of its CUDA graph)
struct PostArgs {
    const float *heat, *paf;            // float32 device inputs of stages 1-3
    const void *heat_host, *paf_host;   // host inputs to copy in first (nullptr: the device pointers are the caller's)
    size_t h2d_heat_bytes, h2d_paf_bytes;
    const void *heat16, *paf16;         // 16-bit device inputs widened into heat / paf first (EKP_DTYPE_BF16 / EKP_DTYPE_F16)
    int dtype;
    int n, h, w, layout, frontend;
    float thr;
    float *heat_mat, *paf_mat;
};
static bool same_args(const PostArgs& a, const PostArgs& b) {
    return a.heat == b.heat && a.paf == b.paf && a.heat_host == b.heat_host && a.paf_host == b.paf_host && a.heat16 == b.heat16 &&
           a.paf16 == b.paf16 && a.dtype == b.dtype && a.n == b.n && a.h == b.h &&
           a.w == b.w && a.layout == b.layout && a.frontend == b.frontend && memcmp(&a.thr, &b.thr, sizeof(float)) == 0 &&
           a.heat_mat == b.heat_mat && a.paf_mat == b.paf_mat;
}

// host_epoch: g_host_frees when a graph with host inputs was captured.  Its copy nodes refer to the pinned allocation that
// held them; once any block is released by ekp_host_free a new block may come back at the same address, so such graphs
// are not replayed across an ekp_host_free (they would copy from the released allocation).
struct GraphEntry { PostArgs key; cudaGraphExec_t exec; int kernels; unsigned long long stamp, host_epoch; };
static std::atomic<unsigned long long> g_host_frees{0};

struct ekp_ctx {
    int device = 0, max_batch = 0, max_h = 0, max_w = 0, max_peaks = 0, max_humans = 0;
    int max_part = EKP_MAX_PART, max_cand = EKP_MAX_CAND;  // peaks of one part / passing candidates of one limb, per image
    // device work buffers
    RawPeak* raw = nullptr;
    int* raw_count = nullptr;       // [max_batch]
    unsigned* overflow = nullptr;   // [max_batch]  (contiguous with raw_count: one memset)
    ekp_peak* line = nullptr;       // [max_batch][max_peaks]
    int* part_off = nullptr;        // [max_batch][20]
    int* n_peaks = nullptr;         // [max_batch]
    Conn* conns = nullptr;          // [max_batch][19][max_part]
    int* n_conns = nullptr;         // [max_batch][19]
    unsigned char* records = nullptr;  // [max_batch] packed result records (ResultLayout)
    const unsigned char* last_records = nullptr;  // where the last run's assembly wrote them (records, or pinned host)
    int map_h = 0, map_w = 0;       // the last run's full-resolution map, by which ekp_draw_humans normalises
    unsigned* draw_keys = nullptr;  // ekp_draw_humans' per-pixel keys (lazily, grown on demand)
    size_t draw_keys_cap = 0;       // pixels
    unsigned draw_epoch = 0;        // draws since the keys were last cleared (the high 16 bits of every key)
    ResultLayout lay = {};
    float* in_block = nullptr;      // staging for the host-buffer entry point: [heat | paf] of one batch, contiguous
                                    // (also where 16-bit inputs are widened to)
    void* in_block16 = nullptr;     // 16-bit [heat | paf] staging of the host-buffer entry point (lazily, half of in_block)
    float* mat_heat = nullptr;      // context-owned operator-surface tensors (host entry, lazily)
    float* mat_paf = nullptr;
    size_t mat_images = 0, mat_hw = 0;
    float* ax = nullptr;            // dense taps for (tab_h, tab_w)
    float* ay = nullptr;
    int tab_h = 0, tab_w = 0;
    float* cubic = nullptr;         // [8][4]
    double* gauss = nullptr;        // [13]
    unsigned long long serial = 0;  // unique per created context (graphs cached outside the context name it)
    void* prep_tab = nullptr;       // resize tables of the input side for (prep_sh, prep_sw, prep_dest)
    int prep_sh = 0, prep_sw = 0, prep_dest = 0, prep_rh = 0, prep_rw = 0;
    // pinned host mirrors of the results
    unsigned char* h_records = nullptr;
    unsigned char* h_records_dev = nullptr;   // the device's view of the pinned h_records (zero-copy result write-out)
    ekp_peak* h_line = nullptr;
    cudaEvent_t done = nullptr;
    cudaStream_t last_stream = nullptr;
    int last_n = 0;
    bool has_run = false;
    long long launches = 0;
    // CUDA graphs of repeated batches (submit_batch)
    std::vector<GraphEntry>* graphs = nullptr;
    cudaStream_t cap_stream = nullptr;
    bool graphs_ok = true;
    unsigned long long graph_clock = 0;
    long long graph_launches = 0;
    // optional per-stage timing: events recorded on the work stream around each stage
    static const int kRing = 64;
    bool timing = false;
    cudaEvent_t tev[kRing][5] = {};
    long long timed_runs = 0;
};

static inline void mark(ekp_ctx* c, int k, cudaStream_t st) {
    if (c->timing) cudaEventRecord(c->tev[c->timed_runs % ekp_ctx::kRing][k], st);
}

static int ctx_free(ekp_ctx* c) {
    if (!c) return EKP_OK;
    cudaSetDevice(c->device);
    void* dev[] = {c->raw, c->raw_count, c->line, c->part_off, c->n_peaks, c->conns, c->n_conns, c->records,
                   c->in_block, c->in_block16, c->mat_heat, c->mat_paf, c->ax, c->ay, c->cubic, c->gauss, c->prep_tab,
                   c->draw_keys};
    for (void* p : dev) if (p) cudaFree(p);
    void* host[] = {c->h_records, c->h_line};
    for (void* p : host) if (p) cudaFreeHost(p);
    if (c->graphs) { for (GraphEntry& e : *c->graphs) cudaGraphExecDestroy(e.exec); delete c->graphs; }
    if (c->cap_stream) cudaStreamDestroy(c->cap_stream);
    if (c->done) cudaEventDestroy(c->done);
    for (auto& row : c->tev) for (cudaEvent_t e : row) if (e) cudaEventDestroy(e);
    delete c;
    return EKP_OK;
}

extern "C" int ekp_create(ekp_ctx** out, int device, int max_batch, int max_h, int max_w, int max_peaks, int max_humans) {
    return ekp_create_ex(out, device, max_batch, max_h, max_w, max_peaks, max_humans, 0, 0);
}

extern "C" int ekp_create_ex(ekp_ctx** out, int device, int max_batch, int max_h, int max_w, int max_peaks, int max_humans,
                             int max_part, int max_cand) {
    if (!out) return fail(EKP_ERR_ARG, "ekp_create: out is NULL");
    *out = nullptr;
    if (max_part <= 0) max_part = EKP_MAX_PART;
    if (max_cand <= 0) max_cand = EKP_MAX_CAND;
    max_cand = (max_cand + 3) & ~3;  // the candidate arrays are read 16 bytes at a time
    if (max_batch < 1 || max_batch > 65535 || max_h < 5 || max_w < 5 || max_peaks < 1 || max_humans < 1 || max_peaks > EKP_LIMIT_PEAKS ||
        max_humans > EKP_LIMIT_HUMANS || max_part < 1 || max_part > EKP_LIMIT_PART || max_cand < 64 || max_cand > EKP_LIMIT_CAND)
        return fail(EKP_ERR_ARG, "ekp_create: bad capacity (batch %d <= 65535, map %dx%d >= 5x5, peaks %d <= %d, humans %d <= %d, "
                    "peaks per part %d <= %d, candidates per limb 64 <= %d <= %d)", max_batch, max_h, max_w, max_peaks, EKP_LIMIT_PEAKS,
                    max_humans, EKP_LIMIT_HUMANS, max_part, EKP_LIMIT_PART, max_cand, EKP_LIMIT_CAND);
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(EKP_ERR_CUDA, "no CUDA device available (%s); this library has no CPU fallback", cudaGetErrorString(e));
    if (device < 0 || device >= ndev) return fail(EKP_ERR_ARG, "ekp_create: device %d of %d", device, ndev);
    CU(cudaSetDevice(device));
    ekp_ctx* c = new ekp_ctx();
    c->device = device; c->max_batch = max_batch; c->max_h = max_h; c->max_w = max_w;
    c->max_peaks = max_peaks; c->max_humans = max_humans; c->max_part = max_part; c->max_cand = max_cand;
    c->graphs = new std::vector<GraphEntry>();
    static std::atomic<unsigned long long> next_serial{1};
    c->serial = next_serial++;
    const size_t B = (size_t) max_batch;
#define DEV_ALLOC(ptr, bytes)                                                     \
    do {                                                                          \
        cudaError_t _e = cudaMalloc((void**) &(ptr), (bytes));                    \
        if (_e != cudaSuccess) { ctx_free(c); return fail(EKP_ERR_CUDA, "cudaMalloc(%zu) for " #ptr ": %s", (size_t) (bytes), cudaGetErrorString(_e)); } \
    } while (0)
#define HOST_ALLOC(ptr, bytes)                                                    \
    do {                                                                          \
        cudaError_t _e = cudaMallocHost((void**) &(ptr), (bytes));                \
        if (_e != cudaSuccess) { ctx_free(c); return fail(EKP_ERR_CUDA, "cudaMallocHost(%zu) for " #ptr ": %s", (size_t) (bytes), cudaGetErrorString(_e)); } \
    } while (0)
    DEV_ALLOC(c->raw, sizeof(RawPeak) * B * max_peaks);
    DEV_ALLOC(c->raw_count, sizeof(int) * 2 * B);
    c->overflow = reinterpret_cast<unsigned*>(c->raw_count + B);
    DEV_ALLOC(c->line, sizeof(ekp_peak) * B * max_peaks);
    DEV_ALLOC(c->part_off, sizeof(int) * B * 20);
    DEV_ALLOC(c->n_peaks, sizeof(int) * B);
    DEV_ALLOC(c->conns, sizeof(Conn) * B * EKP_NUM_LIMB * max_part);
    DEV_ALLOC(c->n_conns, sizeof(int) * B * EKP_NUM_LIMB);
    c->lay.off_subset = 16;
    c->lay.off_hparts = c->lay.off_subset + sizeof(float) * 20 * (size_t) max_humans;
    c->lay.off_hscore = c->lay.off_hparts + sizeof(ekp_peak) * EKP_NUM_PART * (size_t) max_humans;
    c->lay.stride = (c->lay.off_hscore + sizeof(float) * (size_t) max_humans + 15) & ~(size_t) 15;
    DEV_ALLOC(c->records, c->lay.stride * B);
    DEV_ALLOC(c->cubic, sizeof(float) * 32);
    DEV_ALLOC(c->gauss, sizeof(double) * 13);
    HOST_ALLOC(c->h_records, c->lay.stride * B);
    HOST_ALLOC(c->h_line, sizeof(ekp_peak) * B * max_peaks);
    if (cudaHostGetDevicePointer((void**) &c->h_records_dev, c->h_records, 0) != cudaSuccess) { cudaGetLastError(); c->h_records_dev = nullptr; }
    float cubic[32];
    build_cubic_table(cubic);
    e = cudaMemcpy(c->cubic, cubic, sizeof(cubic), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = set_cubic_table(cubic);
    double gauss[13];
    build_scipy_gauss3(gauss);
    if (e == cudaSuccess) e = cudaMemcpy(c->gauss, gauss, sizeof(gauss), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->done, cudaEventDisableTiming);
    if (e == cudaSuccess) e = configure_dense_frontend();
    if (e == cudaSuccess) e = configure_dense_plane(max_h, max_w);
    if (e == cudaSuccess) e = configure_ref_frontend(max_h, max_w);
    if (e == cudaSuccess) {  // taps of interior rows/columns depend only on the phase (D & 7): constant memory
        std::vector<float> t8;
        build_dense_taps(8, t8);
        e = set_interior_taps(t8.data() + 16 * 8);
    }
    if (e == cudaSuccess) e = configure_peaks_sort(max_peaks);
    if (e == cudaSuccess) e = configure_connect(max_part, max_cand);
    if (e == cudaSuccess) e = configure_assemble(max_humans, max_peaks, max_part);
    if (e != cudaSuccess) { ctx_free(c); return fail(EKP_ERR_CUDA, "context setup: %s", cudaGetErrorString(e)); }
    *out = c;
    return EKP_OK;
}

extern "C" void ekp_destroy(ekp_ctx* ctx) { ctx_free(ctx); }
extern "C" int ekp_last_batch(const ekp_ctx* c) { return c && c->has_run ? c->last_n : 0; }
extern "C" int ekp_max_batch(const ekp_ctx* c) { return c ? c->max_batch : 0; }
extern "C" int ekp_max_peaks(const ekp_ctx* c) { return c ? c->max_peaks : 0; }
extern "C" int ekp_max_humans(const ekp_ctx* c) { return c ? c->max_humans : 0; }
extern "C" int ekp_max_part(const ekp_ctx* c) { return c ? c->max_part : 0; }
extern "C" int ekp_max_cand(const ekp_ctx* c) { return c ? c->max_cand : 0; }
extern "C" long long ekp_kernel_launches(const ekp_ctx* c) { return c ? c->launches : 0; }
extern "C" long long ekp_graph_launches(const ekp_ctx* c) { return c ? c->graph_launches : 0; }

// Pinned host memory for the host-buffer entry point: one block that holds a batch's heat tensor directly followed by
// its PAF tensor arrives on the device with ONE copy.  write_combined != 0 asks for write-combined memory (the CPU must
// only write it, sequentially; reads are uncached and slow).
extern "C" int ekp_host_alloc(void** out, size_t bytes, int write_combined) {
    if (!out || bytes == 0) return fail(EKP_ERR_ARG, "ekp_host_alloc: bad arguments");
    *out = nullptr;
    CU(cudaHostAlloc(out, bytes, write_combined ? cudaHostAllocWriteCombined : cudaHostAllocDefault));
    return EKP_OK;
}
extern "C" int ekp_host_free(void* p) {
    if (p) CU(cudaFreeHost(p));
    g_host_frees.fetch_add(1, std::memory_order_acq_rel);
    return EKP_OK;
}

static int ensure_tables(ekp_ctx* c, int h, int w, cudaStream_t stream) {
    if (c->tab_h == h && c->tab_w == w) return EKP_OK;
    std::vector<float> tx, ty;
    if (build_dense_taps(w, tx) || build_dense_taps(h, ty)) return fail(EKP_ERR_ARG, "dense front-end needs h, w >= 5 (got %dx%d)", h, w);
    {   // the kernel reads interior row blocks (2 <= m <= h-3) from the phase table in constant memory
        std::vector<float> t8;
        build_dense_taps(8, t8);
        for (int Y = 16; Y < 8 * (h - 2); Y++)
            if (memcmp(&ty[(size_t) Y * 8], &t8[(size_t) (16 + (Y & 7)) * 8], 8 * sizeof(float)) != 0)
                return fail(EKP_ERR_STATE, "internal: interior taps are not periodic at row %d", Y);
    }
    CU(cudaStreamSynchronize(stream));  // nothing in flight may still read the old tables
    if (c->has_run) CU(cudaEventSynchronize(c->done));
    for (GraphEntry& e : *c->graphs) cudaGraphExecDestroy(e.exec);  // captured with the old table pointers
    c->graphs->clear();
    if (c->ax) { cudaFree(c->ax); c->ax = nullptr; }
    if (c->ay) { cudaFree(c->ay); c->ay = nullptr; }
    c->tab_h = c->tab_w = 0;
    CU(cudaMalloc((void**) &c->ax, tx.size() * sizeof(float)));
    CU(cudaMalloc((void**) &c->ay, ty.size() * sizeof(float)));
    CU(cudaMemcpy(c->ax, tx.data(), tx.size() * sizeof(float), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(c->ay, ty.data(), ty.size() * sizeof(float), cudaMemcpyHostToDevice));
    c->tab_h = h; c->tab_w = w;
    return EKP_OK;
}

static int check_shape(const ekp_ctx* c, int n, int h, int w, int layout, const char* who) {
    if (!c) return fail(EKP_ERR_ARG, "%s: NULL context", who);
    if (n < 1 || n > c->max_batch) return fail(EKP_ERR_ARG, "%s: batch %d outside [1, %d]", who, n, c->max_batch);
    if (h < 5 || w < 5 || h > c->max_h || w > c->max_w)
        return fail(EKP_ERR_ARG, "%s: stride-8 map %dx%d outside [5x5, %dx%d]", who, h, w, c->max_h, c->max_w);
    if (8 * h > 65535 || 8 * w > 65535) return fail(EKP_ERR_ARG, "%s: full-resolution map larger than 65535", who);
    if (layout != EKP_LAYOUT_NCHW && layout != EKP_LAYOUT_NHWC) return fail(EKP_ERR_ARG, "%s: layout %d", who, layout);
    return EKP_OK;
}

// stages 4-5 + result copies, shared by every entry point
static int run_peak_sort(ekp_ctx* c, int n, int id_from_key, cudaStream_t st) {
    mark(c, 1, st);
    CU(launch_peaks_sort(c->raw, c->raw_count, c->max_peaks, c->max_part, id_from_key, n, c->line, c->part_off, c->n_peaks, c->overflow, st));
    c->launches += 1;
    return EKP_OK;
}
// records_direct: device-visible pinned host memory the assembly writes the result records to itself (no D2H copy node)
static int run_connect_assemble(ekp_ctx* c, int n, const PafSource& paf, int h1, cudaStream_t st, unsigned char* records_direct = nullptr) {
    mark(c, 2, st);
    AsmParams ap;
    ap.line = c->line; ap.max_peaks = c->max_peaks; ap.n_peaks = c->n_peaks; ap.part_off = c->part_off; ap.conns = c->conns;
    ap.n_conns = c->n_conns; ap.max_part = c->max_part; ap.max_humans = c->max_humans; ap.conn_cap = 0; ap.overflow = c->overflow;
    ap.records = records_direct ? records_direct : c->records; ap.lay = c->lay;
    c->last_records = ap.records;
    ConnectParams cp;
    cp.line = c->line; cp.part_off = c->part_off; cp.max_peaks = c->max_peaks; cp.max_part = c->max_part; cp.max_cand = c->max_cand;
    cp.paf = paf; cp.h1 = h1; cp.conns = c->conns; cp.n_conns = c->n_conns; cp.overflow = c->overflow;
    CU(launch_paf_connect(cp, n, st));
    mark(c, 3, st);
    CU(launch_assemble(ap, n, st));
    mark(c, 4, st);
    if (c->timing) c->timed_runs++;
    c->launches += 2;
    if (!records_direct) CU(cudaMemcpyAsync(c->h_records, c->records, c->lay.stride * (size_t) n, cudaMemcpyDeviceToHost, st));  // one packed copy
    return EKP_OK;
}
// after a batch has been put on `st` (eagerly or as a graph launch): results become readable when `done` fires
static int finish_submit(ekp_ctx* c, int n, cudaStream_t st) {
    CU(cudaEventRecord(c->done, st));
    c->last_stream = st; c->last_n = n; c->has_run = true;
    return EKP_OK;
}
static int run_back_half(ekp_ctx* c, int n, int id_from_key, const PafSource& paf, int h1, cudaStream_t st) {
    int rc = run_peak_sort(c, n, id_from_key, st);
    if (rc) return rc;
    return run_connect_assemble(c, n, paf, h1, st);
}

// ---- one batch, stages 1-5 ------------------------------------------------------------------------------------
// Everything one batch puts on a stream: input copies (host entry), counters, the kernels of stages 1-5 and the one packed
// device-to-host copy of the result records.  Issued eagerly or into a stream capture; returns the kernels launched.
static int enqueue_batch(ekp_ctx* c, const PostArgs& a, cudaStream_t st, int* kernels) {
    int k = 0;
    const bool wide = a.dtype == EKP_DTYPE_F32;
    if (a.heat_host) {
        // the copies land where the kernels read: the float32 block, or the 16-bit block that is widened into it below
        char* dh = static_cast<char*>(const_cast<void*>(wide ? static_cast<const void*>(a.heat) : a.heat16));
        char* dp = static_cast<char*>(const_cast<void*>(wide ? static_cast<const void*>(a.paf) : a.paf16));
        // one copy when the caller's two tensors are adjacent in host memory (one pinned block: heat, then paf), else two
        if (static_cast<const char*>(a.heat_host) + a.h2d_heat_bytes == static_cast<const char*>(a.paf_host) && dh + a.h2d_heat_bytes == dp) {
            CU(cudaMemcpyAsync(dh, a.heat_host, a.h2d_heat_bytes + a.h2d_paf_bytes, cudaMemcpyHostToDevice, st));
        } else {
            CU(cudaMemcpyAsync(dh, a.heat_host, a.h2d_heat_bytes, cudaMemcpyHostToDevice, st));
            CU(cudaMemcpyAsync(dp, a.paf_host, a.h2d_paf_bytes, cudaMemcpyHostToDevice, st));
        }
    }
    CU(cudaMemsetAsync(c->raw_count, 0, sizeof(int) * 2 * (size_t) c->max_batch, st));
    mark(c, 0, st);
    if (!wide) {
        const size_t px = (size_t) a.n * a.h * a.w;
        CU(launch_widen(a.heat16, a.paf16, px * EKP_HEAT_CH, px * EKP_PAF_CH, a.dtype, const_cast<float*>(a.heat), const_cast<float*>(a.paf), st));
        k += 1;
    }
    PafSource src;
    src.layout = a.layout; src.H = 8 * a.h; src.W = 8 * a.w; src.C = EKP_PAF_CH; src.h = a.h; src.w = a.w;
    src.pair_base = nullptr; src.ids_are_rows = 1;
    if (a.frontend == EKP_FRONTEND_DENSE) {
        DenseParams p;
        p.heat = a.heat; p.paf = a.paf; p.n = a.n; p.h = a.h; p.w = a.w; p.layout = a.layout; p.thr = a.thr;
        p.ax = c->ax; p.ay = c->ay; p.heat_mat = a.heat_mat; p.paf_mat = a.paf_mat; p.smooth_out = nullptr;
        p.raw = c->raw; p.raw_count = c->raw_count; p.raw_cap = c->max_peaks; p.tile_wl = dense_frontend_tile_wl(a.w);
        CU(launch_dense_frontend(p, st));
        k += 1;
        // Stage 4 evaluates the bilinear expression of the materialising kernel on the stride-8 PAF (bit-identical to
        // reading the materialised paf_mat[y][x], tests/test_gpu_parity.py: lean == materialised): the stride-8 planes
        // are L2-resident, while gathers from the 36 MB-per-image paf_mat go to DRAM.
        // EKP_CONNECT_FROM_MAT=1 reads paf_mat instead, exactly as the reference's process_paf does.
        static const bool from_mat = getenv("EKP_CONNECT_FROM_MAT") && atoi(getenv("EKP_CONNECT_FROM_MAT")) != 0;
        if (a.paf_mat && from_mat) { src.ptr = a.paf_mat; src.mode = PAF_FULL_HWC; }
        else { src.ptr = a.paf; src.mode = PAF_LO_BILINEAR; }
    } else {
        RefParams p;
        p.heat = a.heat; p.n = a.n; p.h = a.h; p.w = a.w; p.layout = a.layout; p.thr = a.thr;
        p.raw = c->raw; p.raw_count = c->raw_count; p.raw_cap = c->max_peaks; p.cubic = c->cubic;
        p.gauss = c->gauss;
        p.refine = a.frontend == EKP_FRONTEND_REFERENCE ? 1 : (a.frontend == EKP_FRONTEND_REFERENCE_GAUSS ? 2 : 0);
        CU(launch_ref_frontend(p, st));
        k += ref_frontend_launches(p.refine);
        if (a.paf_mat) { CU(launch_upsample_nearest(a.paf, a.layout, a.n, a.h, a.w, EKP_PAF_CH, a.paf_mat, st)); k += 1; }
        if (a.heat_mat) { CU(launch_upsample_nearest(a.heat, a.layout, a.n, a.h, a.w, EKP_HEAT_CH, a.heat_mat, st)); k += 1; }
        src.ptr = a.paf; src.mode = PAF_LO_NEAREST;  // == paf_mat[y][x] exactly (cv2 INTER_NEAREST x8)
    }
    const long long before = c->launches;
    int rc = run_back_half(c, a.n, /*id_from_key=*/0, src, /*h1=*/8 * a.h, st);
    if (rc) return rc;
    k += (int) (c->launches - before);
    c->launches = before;  // the caller accounts for the whole batch
    *kernels = k;
    return EKP_OK;
}

// A batch with the same pointers, shape and flags as an earlier one (a stream of frames through the same buffers)
// is replayed as a CUDA graph: one launch call instead of nine stream operations, and no gaps between the small
// latency-bound kernels of stages 4-5.  EKP_GRAPHS=0 keeps everything eager (as does per-stage timing).
static const size_t kMaxGraphs = 8;

static int submit_batch(ekp_ctx* c, const PostArgs& a, cudaStream_t st) {
    if (c->has_run && c->last_stream != st) CU(cudaStreamWaitEvent(st, c->done, 0));  // the work buffers are per context
    int kernels = 0;
    static const bool graphs_off = getenv("EKP_GRAPHS") && atoi(getenv("EKP_GRAPHS")) == 0;
    const bool use_graph = !graphs_off && !c->timing && c->graphs_ok;
    if (!use_graph) {
        int rc = enqueue_batch(c, a, st, &kernels);
        if (rc) return rc;
        c->launches += kernels;
    } else {
        std::vector<GraphEntry>& G = *c->graphs;
        GraphEntry* hit = nullptr;
        const unsigned long long epoch = a.heat_host ? g_host_frees.load(std::memory_order_acquire) : 0;
        for (size_t i = 0; i < G.size(); i++) {
            if (!same_args(G[i].key, a)) continue;
            if (G[i].host_epoch == epoch) { hit = &G[i]; break; }
            cudaGraphExecDestroy(G[i].exec);  // captured before a host block was released: capture again
            G.erase(G.begin() + (long) i);
            break;
        }
        if (!hit) {
            if (!c->cap_stream) CU(cudaStreamCreateWithFlags(&c->cap_stream, cudaStreamNonBlocking));
            cudaGraph_t graph = nullptr;
            CU(cudaStreamBeginCapture(c->cap_stream, cudaStreamCaptureModeThreadLocal));
            int rc = enqueue_batch(c, a, c->cap_stream, &kernels);
            cudaError_t ce = cudaStreamEndCapture(c->cap_stream, &graph);
            cudaGraphExec_t exec = nullptr;
            if (rc == EKP_OK && ce == cudaSuccess && graph) ce = cudaGraphInstantiate(&exec, graph, 0);
            if (graph) cudaGraphDestroy(graph);
            if (rc != EKP_OK || ce != cudaSuccess || !exec) {  // no graph on this driver / for this sequence: stay eager from now on
                cudaGetLastError();
                c->graphs_ok = false;
                return submit_batch(c, a, st);
            }
            if (G.size() >= kMaxGraphs) {  // evict the least recently used
                size_t lru = 0;
                for (size_t i = 1; i < G.size(); i++) if (G[i].stamp < G[lru].stamp) lru = i;
                cudaGraphExecDestroy(G[lru].exec);
                G.erase(G.begin() + (long) lru);
            }
            G.push_back(GraphEntry{a, exec, kernels, 0, epoch});
            hit = &G.back();
        }
        hit->stamp = ++c->graph_clock;
        CU(cudaGraphLaunch(hit->exec, st));
        c->launches += hit->kernels;
        c->graph_launches += 1;
    }
    c->map_h = 8 * a.h; c->map_w = 8 * a.w;
    return finish_submit(c, a.n, st);
}

static int check_post_args(const ekp_ctx* c, int n, int h, int w, int layout, int frontend, const char* who) {
    int rc = check_shape(c, n, h, w, layout, who);
    if (rc) return rc;
    if (frontend != EKP_FRONTEND_DENSE && frontend != EKP_FRONTEND_REFERENCE && frontend != EKP_FRONTEND_REFERENCE_COARSE &&
        frontend != EKP_FRONTEND_REFERENCE_GAUSS)
        return fail(EKP_ERR_ARG, "%s: frontend %d", who, frontend);
    return EKP_OK;
}

static int check_dtype(int dtype, const void* heat, const void* paf, const char* who) {
    if (dtype != EKP_DTYPE_F32 && dtype != EKP_DTYPE_BF16 && dtype != EKP_DTYPE_F16)
        return fail(EKP_ERR_ARG, "%s: dtype %d (EKP_DTYPE_F32 0, EKP_DTYPE_BF16 1, EKP_DTYPE_F16 2)", who, dtype);
    if (dtype != EKP_DTYPE_F32 && ((reinterpret_cast<uintptr_t>(heat) | reinterpret_cast<uintptr_t>(paf)) & 1u))
        return fail(EKP_ERR_ARG, "%s: 16-bit heat / paf must be 2-byte aligned", who);
    return EKP_OK;
}

// the context's float32 input block [heat | paf] (host entry: the copy target; 16-bit inputs: the widening target)
static int ensure_in_block(ekp_ctx* c) {
    if (!c->in_block)  // ONE staging block: heat, directly followed by paf (so adjacent host tensors arrive with one copy)
        CU(cudaMalloc((void**) &c->in_block, sizeof(float) * (size_t) c->max_batch * c->max_h * c->max_w * (EKP_HEAT_CH + EKP_PAF_CH)));
    return EKP_OK;
}

static int postprocess_dev(ekp_ctx* c, const void* heat, const void* paf, int dtype, int n, int h, int w, int layout, float thr_heat,
                           int frontend, float* heat_mat, float* paf_mat, void* stream, const char* who) {
    int rc = check_post_args(c, n, h, w, layout, frontend, who);
    if (rc) return rc;
    if (!heat || !paf) return fail(EKP_ERR_ARG, "%s: NULL input", who);
    rc = check_dtype(dtype, heat, paf, who);
    if (rc) return rc;
    if (heat_mat && !paf_mat) return fail(EKP_ERR_ARG, "%s: heat_mat without paf_mat", who);
    if ((reinterpret_cast<uintptr_t>(heat_mat) | reinterpret_cast<uintptr_t>(paf_mat)) & 15u)
        return fail(EKP_ERR_ARG, "%s: heat_mat / paf_mat must be 16-byte aligned (they are written with 16-byte bulk copies)", who);
    if (dtype == EKP_DTYPE_F32 && ((reinterpret_cast<uintptr_t>(heat) | reinterpret_cast<uintptr_t>(paf)) & 3u))
        return fail(EKP_ERR_ARG, "%s: heat / paf must be 4-byte aligned", who);
    cudaStream_t st = (cudaStream_t) stream;
    CU(cudaSetDevice(c->device));
    if (frontend == EKP_FRONTEND_DENSE) {
        rc = ensure_tables(c, h, w, st);
        if (rc) return rc;
    }
    PostArgs a = {};
    a.dtype = dtype;
    if (dtype == EKP_DTYPE_F32) {
        a.heat = static_cast<const float*>(heat); a.paf = static_cast<const float*>(paf);
    } else {
        rc = ensure_in_block(c);
        if (rc) return rc;
        a.heat16 = heat; a.paf16 = paf;
        a.heat = c->in_block; a.paf = c->in_block + (size_t) n * h * w * EKP_HEAT_CH;
    }
    a.n = n; a.h = h; a.w = w; a.layout = layout; a.frontend = frontend; a.thr = thr_heat;
    a.heat_mat = heat_mat; a.paf_mat = paf_mat;
    return submit_batch(c, a, st);
}

static int postprocess_host(ekp_ctx* c, const void* heat_host, const void* paf_host, int dtype, int n, int h, int w, int layout,
                            float thr_heat, int frontend, int materialize, void* stream, const char* who) {
    int rc = check_post_args(c, n, h, w, layout, frontend, who);
    if (rc) return rc;
    if (!heat_host || !paf_host) return fail(EKP_ERR_ARG, "%s: NULL input", who);
    rc = check_dtype(dtype, heat_host, paf_host, who);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t) stream;
    CU(cudaSetDevice(c->device));
    rc = ensure_in_block(c);
    if (rc) return rc;
    if (dtype != EKP_DTYPE_F32 && !c->in_block16)  // the 16-bit copy target, laid out like in_block
        CU(cudaMalloc(&c->in_block16, 2 * (size_t) c->max_batch * c->max_h * c->max_w * (EKP_HEAT_CH + EKP_PAF_CH)));
    const size_t hw = (size_t) h * w;
    float *hm = nullptr, *pm = nullptr;
    if (materialize) {
        if (c->mat_images < (size_t) n || c->mat_hw < hw) {
            CU(cudaStreamSynchronize(st));
            if (c->has_run) CU(cudaEventSynchronize(c->done));
            for (GraphEntry& e : *c->graphs) cudaGraphExecDestroy(e.exec);  // they point at the old tensors
            c->graphs->clear();
            if (c->mat_heat) { cudaFree(c->mat_heat); c->mat_heat = nullptr; }
            if (c->mat_paf) { cudaFree(c->mat_paf); c->mat_paf = nullptr; }
            c->mat_images = 0; c->mat_hw = 0;
            const size_t ni = (size_t) n;
            CU(cudaMalloc((void**) &c->mat_heat, sizeof(float) * ni * hw * 64 * EKP_HEAT_CH));
            CU(cudaMalloc((void**) &c->mat_paf, sizeof(float) * ni * hw * 64 * EKP_PAF_CH));
            c->mat_images = ni; c->mat_hw = hw;
        }
        hm = c->mat_heat; pm = c->mat_paf;
    }
    if (frontend == EKP_FRONTEND_DENSE) {
        rc = ensure_tables(c, h, w, st);
        if (rc) return rc;
    }
    const size_t elem = dtype == EKP_DTYPE_F32 ? sizeof(float) : 2;
    PostArgs a = {};
    a.heat_host = heat_host; a.paf_host = paf_host; a.dtype = dtype;
    a.h2d_heat_bytes = elem * (size_t) n * hw * EKP_HEAT_CH;
    a.h2d_paf_bytes = elem * (size_t) n * hw * EKP_PAF_CH;
    a.heat = c->in_block; a.paf = c->in_block + (size_t) n * hw * EKP_HEAT_CH;
    if (dtype != EKP_DTYPE_F32) { a.heat16 = c->in_block16; a.paf16 = static_cast<char*>(c->in_block16) + a.h2d_heat_bytes; }
    a.n = n; a.h = h; a.w = w; a.layout = layout; a.frontend = frontend; a.thr = thr_heat; a.heat_mat = hm; a.paf_mat = pm;
    return submit_batch(c, a, st);
}

extern "C" int ekp_postprocess(ekp_ctx* c, const float* heat, const float* paf, int n, int h, int w, int layout,
                               float thr_heat, int frontend, float* heat_mat, float* paf_mat, void* stream) {
    return postprocess_dev(c, heat, paf, EKP_DTYPE_F32, n, h, w, layout, thr_heat, frontend, heat_mat, paf_mat, stream, "ekp_postprocess");
}

extern "C" int ekp_postprocess_typed(ekp_ctx* c, const void* heat, const void* paf, int dtype, int n, int h, int w, int layout,
                                     float thr_heat, int frontend, float* heat_mat, float* paf_mat, void* stream) {
    return postprocess_dev(c, heat, paf, dtype, n, h, w, layout, thr_heat, frontend, heat_mat, paf_mat, stream, "ekp_postprocess_typed");
}

extern "C" int ekp_postprocess_host(ekp_ctx* c, const float* heat_host, const float* paf_host, int n, int h, int w,
                                    int layout, float thr_heat, int frontend, int materialize, void* stream) {
    return postprocess_host(c, heat_host, paf_host, EKP_DTYPE_F32, n, h, w, layout, thr_heat, frontend, materialize, stream,
                            "ekp_postprocess_host");
}

extern "C" int ekp_postprocess_host_typed(ekp_ctx* c, const void* heat_host, const void* paf_host, int dtype, int n, int h, int w,
                                          int layout, float thr_heat, int frontend, int materialize, void* stream) {
    return postprocess_host(c, heat_host, paf_host, dtype, n, h, w, layout, thr_heat, frontend, materialize, stream,
                            "ekp_postprocess_host_typed");
}

extern "C" int ekp_process_paf_dev(ekp_ctx* c, const float* peaks, const int* n_peaks, int peaks_stride, int n, int h1,
                                   const float* paf_mat, int H, int W, int C, void* stream) {
    if (!c) return fail(EKP_ERR_ARG, "ekp_process_paf_dev: NULL context");
    if (n < 1 || n > c->max_batch) return fail(EKP_ERR_ARG, "ekp_process_paf_dev: batch %d outside [1, %d]", n, c->max_batch);
    if (!peaks || !paf_mat || !n_peaks) return fail(EKP_ERR_ARG, "ekp_process_paf_dev: NULL input");
    if (H < 1 || W < 1 || C < 38 || peaks_stride < 1) return fail(EKP_ERR_ARG, "ekp_process_paf_dev: bad dims H=%d W=%d C=%d (C >= 38)", H, W, C);
    cudaStream_t st = (cudaStream_t) stream;
    CU(cudaSetDevice(c->device));
    if (c->has_run && c->last_stream != st) CU(cudaStreamWaitEvent(st, c->done, 0));
    CU(cudaMemsetAsync(c->raw_count, 0, sizeof(int) * 2 * (size_t) c->max_batch, st));
    mark(c, 0, st);
    CU(launch_peaks_ingest(peaks, n_peaks, 0, peaks_stride, 5, n, W, H, c->raw, c->raw_count, c->max_peaks, c->overflow, st));
    c->launches += 1;
    PafSource src;
    src.ptr = paf_mat; src.mode = PAF_FULL_HWC; src.layout = EKP_LAYOUT_NHWC; src.H = H; src.W = W; src.C = C; src.h = H / 8; src.w = W / 8;
    src.pair_base = nullptr; src.ids_are_rows = 0;
    int rc = run_back_half(c, n, /*id_from_key=*/1, src, h1, st);
    if (rc) return rc;
    c->map_h = H; c->map_w = W;
    return finish_submit(c, n, st);
}

static int wait_results(ekp_ctx* c, const char* who) {
    if (!c) return fail(EKP_ERR_ARG, "%s: NULL context", who);
    if (!c->has_run) return fail(EKP_ERR_STATE, "%s: no run has been submitted on this context", who);
    CU(cudaSetDevice(c->device));
    CU(cudaEventSynchronize(c->done));
    return EKP_OK;
}
struct RecHead { int num_humans, n_peaks; unsigned overflow; int pad; };
static const RecHead* rec_head(const ekp_ctx* c, int i) { return reinterpret_cast<const RecHead*>(c->h_records + c->lay.stride * (size_t) i); }

static int overflow_status(const ekp_ctx* c) {
    unsigned any = 0;
    for (int i = 0; i < c->last_n; i++) any |= rec_head(c, i)->overflow;
    if (any & EKP_OVF_BADPEAK) return fail(EKP_ERR_ARG, "a peak has part id outside [0,18), coordinates outside the PAF map, or a NaN score");
    if (any) return fail(EKP_ERR_CAPACITY, "capacity overflow (bits 0x%x: 1 peaks>%d, 2 part>%d, 4 candidates>%d, 8 humans>%d)", any,
                         c->max_peaks, c->max_part, c->max_cand, c->max_humans);
    return EKP_OK;
}

extern "C" int ekp_results(ekp_ctx* c, int* num_humans, float* subset, int* n_peaks, ekp_peak* peaks_line, unsigned* overflow) {
    int rc = wait_results(c, "ekp_results");
    if (rc) return rc;
    const int n = c->last_n;
    const size_t mh = (size_t) c->max_humans;
    for (int i = 0; i < n; i++) {
        const RecHead* hd = rec_head(c, i);
        if (num_humans) num_humans[i] = hd->num_humans;
        if (n_peaks) n_peaks[i] = hd->n_peaks;
        if (overflow) overflow[i] = hd->overflow;
        if (subset) memcpy(subset + (size_t) i * mh * 20, c->h_records + c->lay.stride * (size_t) i + c->lay.off_subset,
                           sizeof(float) * 20 * (size_t) hd->num_humans);
    }
    if (peaks_line) {  // the big table is only fetched on request
        CU(cudaMemcpyAsync(c->h_line, c->line, sizeof(ekp_peak) * (size_t) n * c->max_peaks, cudaMemcpyDeviceToHost, c->last_stream));
        CU(cudaStreamSynchronize(c->last_stream));
        for (int i = 0; i < n; i++)  // only the valid rows: what lies behind them in the work buffer is stale
            memcpy(peaks_line + (size_t) i * c->max_peaks, c->h_line + (size_t) i * c->max_peaks,
                   sizeof(ekp_peak) * (size_t) std::min(rec_head(c, i)->n_peaks, c->max_peaks));
    }
    return overflow_status(c);
}

extern "C" int ekp_results_humans(ekp_ctx* c, int* num_humans, ekp_peak* parts, float* scores, unsigned* overflow) {
    int rc = wait_results(c, "ekp_results_humans");
    if (rc) return rc;
    const int n = c->last_n;
    const size_t mh = (size_t) c->max_humans;
    for (int i = 0; i < n; i++) {
        const RecHead* hd = rec_head(c, i);
        const unsigned char* rec = c->h_records + c->lay.stride * (size_t) i;
        if (num_humans) num_humans[i] = hd->num_humans;
        if (overflow) overflow[i] = hd->overflow;
        if (parts) memcpy(parts + (size_t) i * mh * EKP_NUM_PART, rec + c->lay.off_hparts, sizeof(ekp_peak) * EKP_NUM_PART * (size_t) hd->num_humans);
        if (scores) memcpy(scores + (size_t) i * mh, rec + c->lay.off_hscore, sizeof(float) * (size_t) hd->num_humans);
    }
    return overflow_status(c);
}

// ---- drawing (draw.cu) --------------------------------------------------------------------------
extern "C" int ekp_draw_humans(ekp_ctx* c, unsigned char* frames, int n, int H, int W, void* stream) {
    if (!c) return fail(EKP_ERR_ARG, "ekp_draw_humans: NULL context");
    if (!c->has_run) return fail(EKP_ERR_STATE, "ekp_draw_humans: no run has been submitted on this context");
    if (!frames) return fail(EKP_ERR_ARG, "ekp_draw_humans: NULL frames");
    if (n != c->last_n) return fail(EKP_ERR_ARG, "ekp_draw_humans: %d frames for a run of %d images", n, c->last_n);
    if (H < 1 || W < 1 || H > EKP_DRAW_MAX_SIDE || W > EKP_DRAW_MAX_SIDE)
        return fail(EKP_ERR_ARG, "ekp_draw_humans: frame %dx%d outside [1x1, %dx%d]", H, W, EKP_DRAW_MAX_SIDE, EKP_DRAW_MAX_SIDE);
    cudaStream_t st = (cudaStream_t) stream;
    CU(cudaSetDevice(c->device));
    if (c->last_stream != st) CU(cudaStreamWaitEvent(st, c->done, 0));  // the records of the run, the keys of earlier draws
    const size_t pixels = (size_t) n * H * W;
    if (c->draw_keys_cap < pixels) {
        CU(cudaEventSynchronize(c->done));  // no draw in flight may still use the old keys
        if (c->draw_keys) { cudaFree(c->draw_keys); c->draw_keys = nullptr; }
        c->draw_keys_cap = 0;
        CU(cudaMalloc((void**) &c->draw_keys, sizeof(unsigned) * pixels));
        c->draw_keys_cap = pixels;
        c->draw_epoch = 0xffff;  // cleared below
    }
    if (c->draw_epoch == 0xffff) {  // the epoch would wrap: keys of old draws could equal or exceed this draw's
        CU(cudaMemsetAsync(c->draw_keys, 0, sizeof(unsigned) * c->draw_keys_cap, st));
        c->draw_epoch = 0;
    }
    c->draw_epoch += 1;
    CU(launch_draw(c->last_records, c->lay, c->max_humans, c->map_h, c->map_w, frames, n, H, W, c->draw_keys, c->draw_epoch, st));
    c->launches += 2;
    // a later run on any stream waits for this draw before it overwrites the records (submit_batch)
    CU(cudaEventRecord(c->done, st));
    c->last_stream = st;
    return EKP_OK;
}

extern "C" int ekp_debug_raster_host(int kind, int x0, int y0, int x1, int y1, int H, int W, unsigned char* mask) {
    if (!mask || (kind != 1 && kind != 2) || H < 1 || W < 1 || H > EKP_DRAW_MAX_SIDE || W > EKP_DRAW_MAX_SIDE)
        return fail(EKP_ERR_ARG, "ekp_debug_raster_host: bad arguments");
    debug_raster_host(kind, x0, y0, x1, y1, H, W, mask);
    return EKP_OK;
}

extern "C" int ekp_debug_draw_host(const int* num_humans, const ekp_peak* parts, int max_humans, int map_h, int map_w,
                                   unsigned char* frames, int n, int H, int W) {
    if (!num_humans || !parts || !frames || n < 1 || max_humans < 1 || max_humans > EKP_LIMIT_HUMANS || map_h < 1 || map_w < 1 ||
        H < 1 || W < 1 || H > EKP_DRAW_MAX_SIDE || W > EKP_DRAW_MAX_SIDE)
        return fail(EKP_ERR_ARG, "ekp_debug_draw_host: bad arguments");
    debug_draw_host(num_humans, parts, max_humans, map_h, map_w, frames, n, H, W);
    return EKP_OK;
}

extern "C" int ekp_debug_std_sort(ekp_ctx* c, float* scores_dev, unsigned* tags_dev, int n, void* stream) {
    if (!c || n < 0 || (n > 0 && (!scores_dev || !tags_dev))) return fail(EKP_ERR_ARG, "ekp_debug_std_sort: bad arguments");
    if (n == 0) return EKP_OK;
    if (n > 16384) return fail(EKP_ERR_ARG, "ekp_debug_std_sort: n %d > 16384", n);
    if (debug_std_sort_scratch_words(n) * sizeof(unsigned) > sizeof(Conn) * (size_t) c->max_batch * EKP_NUM_LIMB * c->max_part)
        return fail(EKP_ERR_ARG, "ekp_debug_std_sort: n %d needs more scratch than this context's connection buffer holds", n);
    CU(cudaSetDevice(c->device));
    // scratch for the replay's work lists: the connection buffer (idle between runs)
    CU(launch_debug_std_sort(scores_dev, tags_dev, n, reinterpret_cast<unsigned*>(c->conns), (cudaStream_t) stream));
    c->launches += 1;
    return EKP_OK;
}

// ---- input side ---------------------------------------------------------------------------------
extern "C" int ekp_preprocess_dims(int sh, int sw, int dest_size, int factor, int* rh, int* rw, int* ph, int* pw, double* scale) {
    if (sh < 1 || sw < 1 || dest_size < 1 || factor < 1) return fail(EKP_ERR_ARG, "ekp_preprocess_dims: bad arguments");
    const int longest = sh > sw ? sh : sw;
    const double sc = (double) ((float) dest_size) / (double) longest;  // float(dest_size) / im_size_max (estimator.py:59)
    const int r_w = (int) lrint((double) sw * sc), r_h = (int) lrint((double) sh * sc);  // cv2: saturate_cast<int>(size * fx)
    if (rh) *rh = r_h;
    if (rw) *rw = r_w;
    if (ph) *ph = (int) ceil((double) r_h / factor) * factor;
    if (pw) *pw = (int) ceil((double) r_w / factor) * factor;
    if (scale) *scale = sc;
    return EKP_OK;
}

// OpenCV's 11-bit fixed-point bilinear coefficients (resize.cpp): the x axis zeroes the fraction at
// the borders, the y axis keeps it and the kernel clamps the row indices instead.
static void linear_table(int dn, int sn, double scale, bool clamp_frac, int* ofs, short* coef) {
    for (int d = 0; d < dn; d++) {
        volatile float f = (float) (((double) d + 0.5) * scale - 0.5);
        int s = (int) floorf(f);
        f = f - (float) s;
        if (clamp_frac && s < 0) { f = 0.f; s = 0; }
        if (clamp_frac && s >= sn - 1) { f = 0.f; s = sn - 1; }
        ofs[d] = s;
        volatile float w0 = (1.f - f) * 2048.f, w1 = f * 2048.f;
        coef[2 * d] = (short) lrint((double) w0);
        coef[2 * d + 1] = (short) lrint((double) w1);
    }
}

extern "C" int ekp_preprocess(ekp_ctx* c, const unsigned char* frames, int n, int sh, int sw, int dest_size, int factor,
                              int mode, float* out, void* stream) {
    if (!c) return fail(EKP_ERR_ARG, "ekp_preprocess: NULL context");
    if (!frames || !out || n < 1 || (mode != 0 && mode != 1)) return fail(EKP_ERR_ARG, "ekp_preprocess: bad arguments");
    int rh, rw, ph, pw;
    double scale;
    int rc = ekp_preprocess_dims(sh, sw, dest_size, factor, &rh, &rw, &ph, &pw, &scale);
    if (rc) return rc;
    if (rh < 1 || rw < 1) return fail(EKP_ERR_ARG, "ekp_preprocess: image too small");
    cudaStream_t st = (cudaStream_t) stream;
    CU(cudaSetDevice(c->device));
    const size_t tab_bytes = sizeof(int) * ((size_t) rw + rh) + sizeof(short) * 2 * ((size_t) rw + rh);
    if (c->prep_sh != sh || c->prep_sw != sw || c->prep_dest != dest_size) {
        std::vector<int> ofs((size_t) rw + rh);
        std::vector<short> coef(2 * ((size_t) rw + rh));
        linear_table(rw, sw, 1.0 / scale, true, ofs.data(), coef.data());
        linear_table(rh, sh, 1.0 / scale, false, ofs.data() + rw, coef.data() + 2 * (size_t) rw);
        CU(cudaStreamSynchronize(st));
        if (c->prep_tab) { cudaFree(c->prep_tab); c->prep_tab = nullptr; }
        c->prep_sh = c->prep_sw = 0;
        CU(cudaMalloc(&c->prep_tab, tab_bytes));
        CU(cudaMemcpy(c->prep_tab, ofs.data(), sizeof(int) * ofs.size(), cudaMemcpyHostToDevice));
        CU(cudaMemcpy((char*) c->prep_tab + sizeof(int) * ofs.size(), coef.data(), sizeof(short) * coef.size(), cudaMemcpyHostToDevice));
        c->prep_sh = sh; c->prep_sw = sw; c->prep_dest = dest_size; c->prep_rh = rh; c->prep_rw = rw;
    }
    const int* xofs = (const int*) c->prep_tab;
    const int* yofs = xofs + rw;
    const short* ialpha = (const short*) ((const char*) c->prep_tab + sizeof(int) * ((size_t) rw + rh));
    const short* ibeta = ialpha + 2 * (size_t) rw;
    CU(launch_preprocess(frames, out, xofs, ialpha, yofs, ibeta, n, sh, sw, rh, rw, ph, pw, mode, st));
    c->launches += 1;
    return EKP_OK;
}

extern "C" int ekp_set_timing(ekp_ctx* c, int enable) {
    if (!c) return fail(EKP_ERR_ARG, "ekp_set_timing: NULL context");
    CU(cudaSetDevice(c->device));
    if (enable && !c->tev[0][0])
        for (auto& row : c->tev) for (cudaEvent_t& e : row) CU(cudaEventCreate(&e));
    c->timing = enable != 0;
    c->timed_runs = 0;
    return EKP_OK;
}

extern "C" int ekp_stage_times(ekp_ctx* c, float* ms, int* runs) {
    int rc = wait_results(c, "ekp_stage_times");
    if (rc) return rc;
    if (!ms) return fail(EKP_ERR_ARG, "ekp_stage_times: NULL pointer");
    CU(cudaStreamSynchronize(c->last_stream));
    const long long have = c->timed_runs < ekp_ctx::kRing ? c->timed_runs : ekp_ctx::kRing;
    double acc[4] = {0, 0, 0, 0};
    for (long long r = 0; r < have; r++)
        for (int k = 0; k < 4; k++) {
            float t = 0.f;
            CU(cudaEventElapsedTime(&t, c->tev[r][k], c->tev[r][k + 1]));
            acc[k] += t;
        }
    for (int k = 0; k < 4; k++) ms[k] = have ? (float) (acc[k] / (double) have) : 0.f;
    if (runs) *runs = (int) have;
    return EKP_OK;
}

extern "C" int ekp_results_parts(ekp_ctx* c, int* part_off) {
    int rc = wait_results(c, "ekp_results_parts");
    if (rc) return rc;
    if (!part_off) return fail(EKP_ERR_ARG, "ekp_results_parts: NULL pointer");
    std::vector<int> tmp((size_t) c->last_n * 20);
    CU(cudaMemcpyAsync(tmp.data(), c->part_off, sizeof(int) * tmp.size(), cudaMemcpyDeviceToHost, c->last_stream));
    CU(cudaStreamSynchronize(c->last_stream));
    for (int i = 0; i < c->last_n; i++) memcpy(part_off + (size_t) i * 19, tmp.data() + (size_t) i * 20, sizeof(int) * 19);
    return EKP_OK;
}

extern "C" int ekp_dense_smooth_debug(ekp_ctx* c, const float* heat, int n, int h, int w, int layout, float* smooth_out, void* stream) {
    int rc = check_shape(c, n, h, w, layout, "ekp_dense_smooth_debug");
    if (rc) return rc;
    if (!heat || !smooth_out) return fail(EKP_ERR_ARG, "ekp_dense_smooth_debug: NULL pointer");
    cudaStream_t st = (cudaStream_t) stream;
    CU(cudaSetDevice(c->device));
    rc = ensure_tables(c, h, w, st);
    if (rc) return rc;
    CU(cudaMemsetAsync(c->raw_count, 0, sizeof(int) * 2 * (size_t) c->max_batch, st));
    DenseParams p;
    p.heat = heat; p.paf = nullptr; p.n = n; p.h = h; p.w = w; p.layout = layout; p.thr = INFINITY;
    p.ax = c->ax; p.ay = c->ay; p.heat_mat = nullptr; p.paf_mat = nullptr; p.smooth_out = smooth_out;
    p.raw = c->raw; p.raw_count = c->raw_count; p.raw_cap = c->max_peaks; p.tile_wl = dense_frontend_tile_wl(w);
    CU(launch_dense_frontend(p, st));
    c->launches += 1;
    return EKP_OK;
}

// ---- the reference operator surface ------------------------------------------------------------
// Process-global "last result", like the reference's globals (pafprocess.cpp:12-13).
namespace {
std::mutex g_mu;
ekp_ctx* g_ctx = nullptr;
float* g_dev_peaks = nullptr; size_t g_dev_peaks_cap = 0;
float* g_dev_paf = nullptr; size_t g_dev_paf_cap = 0;
// sparse upload: sample offsets (device + pinned host), gathered samples (pinned host + device), pair prefix
unsigned* g_dev_offs = nullptr; unsigned* g_host_offs = nullptr; float2* g_host_samp = nullptr; float2* g_dev_samp = nullptr;
size_t g_samp_cap = 0;
int* g_dev_pair_base = nullptr;
const long long kSparseMaxSamples = 8ll << 20;  // beyond this the whole tensor is uploaded instead
std::vector<float> g_subset;      // [num_humans][20]
std::vector<float> g_hscore;      // [num_humans] subset[18] / subset[19], computed on the device
std::vector<ekp_peak> g_line;     // part-sorted peak table
int g_num_humans = 0;

// The context behind the operator surface: re-created with larger capacities when a scene needs them (the new one
// first, so a failed creation leaves the old one in place), never beyond the library's limits.
int compat_ctx(int need_peaks, int need_humans, int need_part, int need_cand) {
    if (g_ctx && g_ctx->max_peaks >= need_peaks && g_ctx->max_humans >= need_humans && g_ctx->max_part >= need_part &&
        g_ctx->max_cand >= need_cand)
        return EKP_OK;
    int dev = 0;
    if (const char* s = getenv("EKP_DEVICE")) dev = atoi(s);
    int peaks = 1024, humans = 128;
    while (peaks < need_peaks) peaks *= 2;
    while (humans < need_humans) humans *= 2;
    peaks = std::min(peaks, EKP_LIMIT_PEAKS);
    humans = std::min(humans, EKP_LIMIT_HUMANS);
    if (g_ctx) { need_part = std::max(need_part, g_ctx->max_part); need_cand = std::max(need_cand, g_ctx->max_cand); }
    ekp_ctx* fresh = nullptr;
    int rc = ekp_create_ex(&fresh, dev, 1, 8, 8, peaks, humans, std::min(need_part, EKP_LIMIT_PART), std::min(need_cand, EKP_LIMIT_CAND));
    if (rc) return rc;
    if (g_ctx) ekp_destroy(g_ctx);
    g_ctx = fresh;
    return EKP_OK;
}
}  // namespace

// ---- process_paf, small scenes: everything stage 4 needs in ONE upload, no mid-call synchronisation ---------------
// For up to kListedMaxSamples samples the host lists them itself: it buckets the caller's peaks by part (the order of
// the reference's own buckets, pafprocess.cpp:24-43), walks the pairs of every limb in the kernel's order (a outer,
// b inner) and copies the two floats at each of the <= 10 sample positions out of the caller's paf_mat -- the positions
// by the roundpaf arithmetic of pafprocess.cpp:228-233, 240-242, which is index arithmetic on the INPUT, not scoring:
// unit vectors, dot products, both criteria, sort, assignment and assembly all run in the kernels, on these values.
// One pinned block [pair prefix | peaks | samples] -> one H2D copy -> ingest, sort, connect (PAF_PACKED), assemble ->
// one D2H copy of the result record -> one wait.  The part-sorted peak table the getters index (pafprocess.cpp:208-218)
// is the bucket order itself, so it never has to come back from the device.
// Returns 1 when the scene is not eligible (an invalid peak, a part over max_part, too many samples): the general path
// below then runs and reports whatever is wrong.
namespace {
const long long kListedMaxSamples = 64 * 1024;
unsigned char* g_listed_host = nullptr; unsigned char* g_listed_dev = nullptr; size_t g_listed_cap = 0;
enum { TINY_OFF = 0, TINY_ZC = 1, TINY_ZC_GRAPH = 2 };
unsigned char* g_listed_host_dev = nullptr;   // the device's view of g_listed_host
struct TinyGraph { unsigned long long ctx_serial; int p3, f1, f2, f3, h1; size_t bytes; cudaGraphExec_t exec; };
std::vector<TinyGraph> g_tiny;   // under g_mu like everything of the operator surface
bool g_tiny_ok = true;
const int kTinyPeaks = 512;
const long long kTinyMaxSamples = 16384;
void tiny_graphs_clear() {
    for (TinyGraph& e : g_tiny) cudaGraphExecDestroy(e.exec);
    g_tiny.clear();
}
const int kHostPairs[EKP_NUM_LIMB][2] = {{1, 2}, {1, 5}, {2, 3}, {3, 4}, {5, 6}, {6, 7}, {1, 8}, {8, 9}, {9, 10}, {1, 11},
                                         {11, 12}, {12, 13}, {1, 0}, {0, 14}, {14, 16}, {0, 15}, {15, 17}, {2, 16}, {5, 17}};
const int kHostPairsNet[EKP_NUM_LIMB] = {12, 20, 14, 16, 22, 24, 0, 2, 4, 6, 8, 10, 28, 30, 34, 32, 36, 18, 26};  // x channel; y = x + 1

static double now_us() {
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return ts.tv_sec * 1e6 + ts.tv_nsec * 1e-3;
}
int process_paf_listed(ekp_ctx* c, long long npk, int p3, const float* peaks, int h1, int f1, int f2, int f3, const float* pafmap,
                       unsigned* ovf_out) {
    static const bool trace = getenv("EKP_TRACE_PROCESS_PAF") != nullptr;   // phase times on stderr (tools/compat_latency.py)
    const double t0 = trace ? now_us() : 0.0;
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
    int pair_base[32] = {0};
    long long acc = 0;
    for (int l = 0; l < EKP_NUM_LIMB; l++) {
        const size_t nA = bucket[kHostPairs[l][0]].size(), nB = bucket[kHostPairs[l][1]].size();
        if (nA > (size_t) c->max_part || nB > (size_t) c->max_part) return 1;
        pair_base[l] = (int) acc;
        acc += (long long) nA * (long long) nB;
    }
    pair_base[EKP_NUM_LIMB] = (int) acc;
    const long long nsamples = acc * 10;
    if (nsamples > kListedMaxSamples) return 1;
    // Tiny scenes (a handful of people: every frame of an ordinary video).  Such a call used to wait ~25 us for the device-side
    // chain H2D copy -> 3 kernels -> D2H copy -> event after spending ~25 us submitting it (70 us at 3 people).  Here the
    // kernels read the pinned block and write the result record THROUGH PCIe themselves (zero-copy: a few KB, one round trip
    // per kernel), so the chain is the three kernels; and the block has a fixed layout (room for kTinyPeaks peaks, samples
    // rounded up to a size class, the peak count inside), so the launch arguments depend only on (shape, size class) and the
    // three launches are replayed as ONE CUDA graph launch (1.5 us to submit).  Measured, raw call at 3 / 8 people: 70 / 112 us
    // before, 58 / 111 us zero-copy with eager launches, 51 / 103 us as a graph (the copies inside a graph instead: 66 / 116 us;
    // profiles/README.md).  What is left is the latency of the three kernels themselves (~35 us).
    // EKP_PROCESS_PAF_TINY = zerocopy_graph (default) | zerocopy (eager launches; also under EKP_GRAPHS=0) | off.
    static const int tiny_mode = [] {
        const char* e = getenv("EKP_PROCESS_PAF_TINY");
        const bool graphs_off = getenv("EKP_GRAPHS") && atoi(getenv("EKP_GRAPHS")) == 0;
        int m = TINY_ZC_GRAPH;
        if (e) m = !strcmp(e, "zerocopy_graph") ? TINY_ZC_GRAPH : (!strcmp(e, "zerocopy") ? TINY_ZC : TINY_OFF);
        if (graphs_off && m == TINY_ZC_GRAPH) m = TINY_ZC;
        return m;
    }();
    bool tiny = tiny_mode != TINY_OFF && g_tiny_ok && !c->timing && c->h_records_dev && npk <= kTinyPeaks && npk <= peaks_one_max() &&
                nsamples <= kTinyMaxSamples;
    long long samp_class = 2048;
    while (samp_class < nsamples) samp_class *= 2;
    pair_base[31] = (int) npk;
    const size_t off_peaks = sizeof(pair_base);
    const size_t off_samp = (off_peaks + sizeof(float) * (size_t) (tiny ? kTinyPeaks : npk) * p3 + 7) & ~(size_t) 7;
    const size_t bytes = off_samp + sizeof(float2) * (size_t) (tiny ? samp_class : (nsamples > 0 ? nsamples : 1));
    if (g_listed_cap < bytes) {
        tiny_graphs_clear();   // they copy from / to the old blocks
        if (g_listed_host) cudaFreeHost(g_listed_host);
        if (g_listed_dev) cudaFree(g_listed_dev);
        g_listed_host = nullptr; g_listed_dev = nullptr; g_listed_cap = 0;
        const size_t cap = bytes + bytes / 2 + 4096;
        CU(cudaMallocHost((void**) &g_listed_host, cap));
        CU(cudaMalloc((void**) &g_listed_dev, cap));
        if (cudaHostGetDevicePointer((void**) &g_listed_host_dev, g_listed_host, 0) != cudaSuccess) { cudaGetLastError(); g_listed_host_dev = nullptr; }
        g_listed_cap = cap;
    }
    if (!g_listed_host_dev) tiny = false;   // pinned memory the device cannot address (no unified addressing): the copying path
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
    const double t1 = trace ? now_us() : 0.0;
    cudaStream_t st = nullptr;
    if (c->has_run && c->last_stream != st) CU(cudaStreamWaitEvent(st, c->done, 0));
    int rc = EKP_OK;
    PafSource src;
    src.layout = EKP_LAYOUT_NHWC; src.H = f1; src.W = f2; src.C = f3; src.h = f1 / 8; src.w = f2 / 8; src.ids_are_rows = 0;
    src.ptr = reinterpret_cast<const float*>(g_listed_dev + off_samp); src.mode = PAF_PACKED;
    src.pair_base = reinterpret_cast<const int*>(g_listed_dev);
    bool launched = false;
    if (tiny) {
        const bool as_graph = tiny_mode == TINY_ZC_GRAPH;
        unsigned char* blk = g_listed_host_dev;   // the kernels read the pinned block itself
        PafSource tsrc = src;
        tsrc.ptr = reinterpret_cast<const float*>(blk + off_samp);
        tsrc.pair_base = reinterpret_cast<const int*>(blk);
        unsigned char* rec_direct = c->h_records_dev;
        auto enqueue = [&](cudaStream_t q) -> int {   // the three kernels on `q`
            CU(launch_peaks_ingest_sort_one(reinterpret_cast<const float*>(blk + off_peaks), 0, reinterpret_cast<const int*>(blk) + 31, p3, f2, f1,
                                            c->max_peaks, c->max_part, c->line, c->part_off, c->n_peaks, c->raw_count, c->overflow, q));
            return run_connect_assemble(c, 1, tsrc, h1, q, rec_direct);
        };
        if (!as_graph) {
            rc = enqueue(st);
            if (rc) return rc;
            c->launches += 1;
            launched = true;
        } else {
            TinyGraph* hit = nullptr;
            for (size_t i = 0; i < g_tiny.size();) {   // graphs of a context that no longer exists go
                if (g_tiny[i].ctx_serial != c->serial) { cudaGraphExecDestroy(g_tiny[i].exec); g_tiny.erase(g_tiny.begin() + (long) i); }
                else i++;
            }
            for (TinyGraph& e : g_tiny)
                if (e.p3 == p3 && e.f1 == f1 && e.f2 == f2 && e.f3 == f3 && e.h1 == h1 && e.bytes == bytes) hit = &e;
            if (!hit) {
                if (!c->cap_stream) CU(cudaStreamCreateWithFlags(&c->cap_stream, cudaStreamNonBlocking));
                const long long before = c->launches;
                cudaGraph_t graph = nullptr;
                cudaGraphExec_t exec = nullptr;
                CU(cudaStreamBeginCapture(c->cap_stream, cudaStreamCaptureModeThreadLocal));
                const int rc2 = enqueue(c->cap_stream);
                cudaError_t ce = cudaStreamEndCapture(c->cap_stream, &graph);
                if (rc2 == EKP_OK && ce == cudaSuccess && graph) ce = cudaGraphInstantiate(&exec, graph, 0);
                if (graph) cudaGraphDestroy(graph);
                c->launches = before;
                if (rc2 != EKP_OK || ce != cudaSuccess || !exec) { cudaGetLastError(); g_tiny_ok = false; }   // stay on the general path from now on
                else {
                    if (g_tiny.size() >= 8) { cudaGraphExecDestroy(g_tiny.front().exec); g_tiny.erase(g_tiny.begin()); }
                    g_tiny.push_back(TinyGraph{c->serial, p3, f1, f2, f3, h1, bytes, exec});
                    hit = &g_tiny.back();
                }
            }
            if (hit) {
                CU(cudaGraphLaunch(hit->exec, st));
                c->launches += 3;
                c->graph_launches += 1;
                launched = true;
            }
        }
    }
    if (!launched) {
        CU(cudaMemcpyAsync(g_listed_dev, g_listed_host, bytes, cudaMemcpyHostToDevice, st));
        mark(c, 0, st);
        mark(c, 1, st);
        if (npk <= peaks_one_max()) {   // ingest + sort in one block, no counters to clear
            CU(launch_peaks_ingest_sort_one(reinterpret_cast<const float*>(g_listed_dev + off_peaks), (int) npk, nullptr, p3, f2, f1, c->max_peaks,
                                            c->max_part, c->line, c->part_off, c->n_peaks, c->raw_count, c->overflow, st));
            c->launches += 1;
        } else {
            CU(cudaMemsetAsync(c->raw_count, 0, sizeof(int) * 2 * (size_t) c->max_batch, st));
            CU(launch_peaks_ingest(reinterpret_cast<const float*>(g_listed_dev + off_peaks), nullptr, (int) npk, (int) npk, p3, 1, f2, f1, c->raw,
                                   c->raw_count, c->max_peaks, c->overflow, st));
            c->launches += 1;
            rc = run_peak_sort(c, 1, /*id_from_key=*/1, st);
            if (rc) return rc;
        }
        rc = run_connect_assemble(c, 1, src, h1, st);
        if (rc) return rc;
    }
    rc = finish_submit(c, 1, st);
    if (rc) return rc;
    const double t2 = trace ? now_us() : 0.0;
    std::vector<float> subset((size_t) c->max_humans * 20);
    int nh = 0, np = 0;
    rc = ekp_results(c, &nh, subset.data(), &np, nullptr, ovf_out);
    if (rc) return rc;
    if (trace) fprintf(stderr, "process_paf listed: %lld peaks %lld samples | host listing %.1f us, submit %.1f us, wait + results %.1f us\n", npk,
                       nsamples, t1 - t0, t2 - t1, now_us() - t2);
    g_num_humans = nh;
    g_subset.assign(subset.begin(), subset.begin() + (size_t) nh * 20);
    const float* hs = reinterpret_cast<const float*>(c->h_records + c->lay.off_hscore);
    g_hscore.assign(hs, hs + nh);
    g_line.clear();
    g_line.reserve((size_t) npk);
    for (int part = 0; part < EKP_NUM_PART; part++)   // peak_infos_line: the buckets one after the other (pafprocess.cpp:38-43)
        for (int kk : bucket[part]) {
            const float* row = peaks + (size_t) kk * p3;
            ekp_peak pk;
            pk.x = (int) row[0]; pk.y = (int) row[1]; pk.score = row[2]; pk.id = kk;
            g_line.push_back(pk);
        }
    return EKP_OK;
}
}  // namespace

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
    int need_humans = 128, need_part = EKP_MAX_PART, need_cand = EKP_MAX_CAND;
    for (int attempt = 0; attempt < 8; attempt++) {
        int rc = compat_ctx((int) npk, need_humans, need_part, need_cand);
        if (rc) return rc;
        ekp_ctx* c = g_ctx;
        CU(cudaSetDevice(c->device));
        const size_t pk_elems = (size_t) npk * p3, paf_elems = (size_t) f1 * f2 * f3;
        if (g_dev_peaks_cap < pk_elems) { if (g_dev_peaks) cudaFree(g_dev_peaks); g_dev_peaks = nullptr; g_dev_peaks_cap = 0;
            CU(cudaMalloc((void**) &g_dev_peaks, pk_elems * sizeof(float))); g_dev_peaks_cap = pk_elems; }
        cudaStream_t st = nullptr;
        const int npk_i = (int) npk;
        const char* upload_mode = getenv("EKP_PROCESS_PAF_UPLOAD");   // unset or "listed": the small-scene path first
        if ((!upload_mode || strcmp(upload_mode, "listed") == 0) && paf_elems < (1ull << 32)) {
            unsigned ovf = 0;
            rc = process_paf_listed(c, npk, p3, peaks, h1, f1, f2, f3, pafmap, &ovf);
            if (rc == EKP_OK) return EKP_OK;
            if (rc == EKP_ERR_CAPACITY && !(ovf & (EKP_OVF_PEAKS | EKP_OVF_BADPEAK))) {
                bool grew = false, stuck = false;
                if (ovf & EKP_OVF_HUMANS) { if (c->max_humans < EKP_LIMIT_HUMANS) { need_humans = std::min(c->max_humans * 4, EKP_LIMIT_HUMANS); grew = true; } else stuck = true; }
                if (ovf & EKP_OVF_PART) { if (c->max_part < EKP_LIMIT_PART) { need_part = std::min(c->max_part * 4, EKP_LIMIT_PART); grew = true; } else stuck = true; }
                if (ovf & EKP_OVF_CANDIDATES) { if (c->max_cand < EKP_LIMIT_CAND) { need_cand = std::min(c->max_cand * 4, EKP_LIMIT_CAND); grew = true; } else stuck = true; }
                if (grew && !stuck) continue;
            }
            if (rc != 1) return rc;
        }
        // Sparse upload (default): stage 4 reads at most 10 positions of paf_mat per candidate pair, a few KB
        // against the 24 MB tensor.  Pairs per limb follow from the part column of the caller's peaks.
        int pair_base[EKP_NUM_LIMB + 1];
        long long nsamples = 0;
        bool sparse = paf_elems < (1ull << 32);
        if (const char* e = getenv("EKP_PROCESS_PAF_UPLOAD")) sparse = sparse && strcmp(e, "dense") != 0;
        if (sparse) {
            int per_part[EKP_NUM_PART] = {0};
            for (long long k = 0; k < npk; k++) {
                const float pt = peaks[k * p3 + 4];
                const int part = pt > -1.f && pt < (float) EKP_NUM_PART ? (int) pt : -1;  // (int) truncates like the ingest kernel;
                if (part >= 0) per_part[part]++;  // any peak it rejects for another reason fails the whole call (EKP_OVF_BADPEAK)
            }
            static const int pairs[EKP_NUM_LIMB][2] = {{1, 2}, {1, 5}, {2, 3}, {3, 4}, {5, 6}, {6, 7}, {1, 8}, {8, 9}, {9, 10}, {1, 11},
                                                       {11, 12}, {12, 13}, {1, 0}, {0, 14}, {14, 16}, {0, 15}, {15, 17}, {2, 16}, {5, 17}};
            long long acc = 0;
            for (int l = 0; l < EKP_NUM_LIMB; l++) {
                pair_base[l] = (int) acc;
                acc += (long long) std::min(per_part[pairs[l][0]], c->max_part) * std::min(per_part[pairs[l][1]], c->max_part);
            }
            pair_base[EKP_NUM_LIMB] = (int) acc;
            nsamples = acc * 10;
            sparse = nsamples <= kSparseMaxSamples;
        }
        CU(cudaMemcpyAsync(g_dev_peaks, peaks, pk_elems * sizeof(float), cudaMemcpyHostToDevice, st));
        CU(cudaMemsetAsync(c->raw_count, 0, sizeof(int) * 2 * (size_t) c->max_batch, st));
        mark(c, 0, st);
        CU(launch_peaks_ingest(g_dev_peaks, nullptr, npk_i, npk_i, p3, 1, f2, f1, c->raw, c->raw_count, c->max_peaks, c->overflow, st));
        c->launches += 1;
        PafSource src;
        src.layout = EKP_LAYOUT_NHWC; src.H = f1; src.W = f2; src.C = f3; src.h = f1 / 8; src.w = f2 / 8; src.pair_base = nullptr;
        src.ids_are_rows = 0;
        rc = run_peak_sort(c, 1, /*id_from_key=*/1, st);
        if (rc) return rc;
        if (sparse && nsamples > 0) {
            if (g_samp_cap < (size_t) nsamples) {
                if (g_dev_offs) cudaFree(g_dev_offs);
                if (g_dev_samp) cudaFree(g_dev_samp);
                if (g_host_offs) cudaFreeHost(g_host_offs);
                if (g_host_samp) cudaFreeHost(g_host_samp);
                g_dev_offs = nullptr; g_dev_samp = nullptr; g_host_offs = nullptr; g_host_samp = nullptr; g_samp_cap = 0;
                const size_t cap = (size_t) nsamples + (size_t) nsamples / 2 + 1024;
                CU(cudaMalloc((void**) &g_dev_offs, cap * sizeof(unsigned)));
                CU(cudaMalloc((void**) &g_dev_samp, cap * sizeof(float2)));
                CU(cudaMallocHost((void**) &g_host_offs, cap * sizeof(unsigned)));
                CU(cudaMallocHost((void**) &g_host_samp, cap * sizeof(float2)));
                g_samp_cap = cap;
            }
            if (!g_dev_pair_base) CU(cudaMalloc((void**) &g_dev_pair_base, sizeof(int) * (EKP_NUM_LIMB + 1)));
            CU(cudaMemcpyAsync(g_dev_pair_base, pair_base, sizeof(pair_base), cudaMemcpyHostToDevice, st));
            CU(cudaMemsetAsync(g_dev_offs, 0, (size_t) nsamples * sizeof(unsigned), st));  // limbs the kernel skips stay in bounds
            CU(launch_pair_sample_offsets(c->line, c->part_off, g_dev_pair_base, f1, f2, f3, c->max_part, g_dev_offs, st));
            c->launches += 1;
            CU(cudaMemcpyAsync(g_host_offs, g_dev_offs, (size_t) nsamples * sizeof(unsigned), cudaMemcpyDeviceToHost, st));
            CU(cudaStreamSynchronize(st));
            for (long long k = 0; k < nsamples; k++) {  // the gather: a copy, no arithmetic
                const float* q = pafmap + g_host_offs[k];
                g_host_samp[k] = make_float2(q[0], q[1]);
            }
            CU(cudaMemcpyAsync(g_dev_samp, g_host_samp, (size_t) nsamples * sizeof(float2), cudaMemcpyHostToDevice, st));
            src.ptr = reinterpret_cast<const float*>(g_dev_samp); src.mode = PAF_PACKED; src.pair_base = g_dev_pair_base;
        } else {
            if (g_dev_paf_cap < paf_elems) { if (g_dev_paf) cudaFree(g_dev_paf); g_dev_paf = nullptr; g_dev_paf_cap = 0;
                CU(cudaMalloc((void**) &g_dev_paf, paf_elems * sizeof(float))); g_dev_paf_cap = paf_elems; }
            CU(cudaMemcpyAsync(g_dev_paf, pafmap, paf_elems * sizeof(float), cudaMemcpyHostToDevice, st));
            src.ptr = g_dev_paf; src.mode = PAF_FULL_HWC;
        }
        rc = run_connect_assemble(c, 1, src, h1, st);
        if (rc) return rc;
        rc = finish_submit(c, 1, st);
        if (rc) return rc;
        std::vector<ekp_peak> line((size_t) c->max_peaks);
        std::vector<float> subset((size_t) c->max_humans * 20);
        int nh = 0, np = 0;
        unsigned ovf = 0;
        rc = ekp_results(c, &nh, subset.data(), &np, line.data(), &ovf);
        if (rc == EKP_ERR_CAPACITY && !(ovf & (EKP_OVF_PEAKS | EKP_OVF_BADPEAK))) {
            // grow exactly what overflowed, within the library's limits, and run again; at a limit the error stands
            bool grew = false, stuck = false;
            if (ovf & EKP_OVF_HUMANS) { if (c->max_humans < EKP_LIMIT_HUMANS) { need_humans = std::min(c->max_humans * 4, EKP_LIMIT_HUMANS); grew = true; } else stuck = true; }
            if (ovf & EKP_OVF_PART) { if (c->max_part < EKP_LIMIT_PART) { need_part = std::min(c->max_part * 4, EKP_LIMIT_PART); grew = true; } else stuck = true; }
            if (ovf & EKP_OVF_CANDIDATES) { if (c->max_cand < EKP_LIMIT_CAND) { need_cand = std::min(c->max_cand * 4, EKP_LIMIT_CAND); grew = true; } else stuck = true; }
            if (grew && !stuck) continue;
        }
        if (rc) return rc;
        g_num_humans = nh;
        g_subset.assign(subset.begin(), subset.begin() + (size_t) nh * 20);
        const float* hs = reinterpret_cast<const float*>(c->h_records + c->lay.off_hscore);
        g_hscore.assign(hs, hs + nh);
        g_line.assign(line.begin(), line.begin() + np);
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
