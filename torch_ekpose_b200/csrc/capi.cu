// capi.cu -- the C ABI of libekpose_b200.so (include/ekpose_b200.h): context and work buffers, the batched device API,
// results, drawing, the input side and timing.  The reference's process_paf / get_* operator surface on top of the same
// context is in process_paf.cu.
// Host code only orchestrates: every stage of the path runs in the CUDA kernels of this
// directory and there is no CPU implementation to fall back to.
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <vector>

#include "capi.cuh"

using namespace ekp;

// ---- error reporting -------------------------------------------------------------------------
static thread_local char g_err[512] = "";
int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

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
static std::atomic<unsigned long long> g_host_frees{0};  // blocks released by ekp_host_free (GraphEntry::host_epoch)

void drop_graphs(ekp_ctx* c) {
    for (GraphEntry& e : c->graphs) cudaGraphExecDestroy(e.exec);
    c->graphs.clear();
}

// Before a buffer that queued work or a cached graph of the context may use is freed: nothing in flight on `st` or of
// the last run may still read it, and no graph may replay with its address.
static int quiesce(ekp_ctx* c, cudaStream_t st) {
    CU(cudaStreamSynchronize(st));
    if (c->has_run) CU(cudaEventSynchronize(c->done));
    drop_graphs(c);
    return EKP_OK;
}

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
    drop_graphs(c);
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
    int rc = quiesce(c, stream);  // the old tables
    if (rc) return rc;
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

// the dense front-end's parameters for heat [n, h, w] in `layout`: the context's taps and raw-peak buffer, no outputs but the peaks
static DenseParams dense_params(const ekp_ctx* c, const float* heat, int n, int h, int w, int layout) {
    DenseParams p = {};
    p.heat = heat; p.n = n; p.h = h; p.w = w; p.layout = layout;
    p.ax = c->ax; p.ay = c->ay;
    p.raw = c->raw; p.raw_count = c->raw_count; p.raw_cap = c->max_peaks; p.tile_wl = dense_frontend_tile_wl(w);
    return p;
}

int run_peak_sort(ekp_ctx* c, int n, int id_from_key, cudaStream_t st) {
    mark(c, 1, st);
    CU(launch_peaks_sort(c->raw, c->raw_count, c->max_peaks, c->max_part, id_from_key, n, c->line, c->part_off, c->n_peaks, c->overflow, st));
    c->launches += 1;
    return EKP_OK;
}
int run_connect_assemble(ekp_ctx* c, int n, const PafSource& paf, int h1, cudaStream_t st, unsigned char* records_direct) {
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
PafSource paf_source(int mode, const void* ptr, const int* pair_base, int f1, int f2, int f3) {
    PafSource s;
    s.ptr = static_cast<const float*>(ptr); s.mode = mode; s.pair_base = pair_base; s.ids_are_rows = 0;
    s.layout = EKP_LAYOUT_NHWC; s.H = f1; s.W = f2; s.C = f3; s.h = f1 / 8; s.w = f2 / 8;
    return s;
}
int finish_submit(ekp_ctx* c, int n, cudaStream_t st) {
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
// device-to-host copy of the result records.  Issued eagerly or into a stream capture.
static int enqueue_batch(ekp_ctx* c, const PostArgs& a, cudaStream_t st) {
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
        c->launches += 1;
    }
    PafSource src;
    src.layout = a.layout; src.H = 8 * a.h; src.W = 8 * a.w; src.C = EKP_PAF_CH; src.h = a.h; src.w = a.w;
    src.pair_base = nullptr; src.ids_are_rows = 1;
    if (a.frontend == EKP_FRONTEND_DENSE) {
        DenseParams p = dense_params(c, a.heat, a.n, a.h, a.w, a.layout);
        p.paf = a.paf; p.thr = a.thr; p.heat_mat = a.heat_mat; p.paf_mat = a.paf_mat;
        CU(launch_dense_frontend(p, st));
        c->launches += 1;
        // Stage 4 evaluates the bilinear expression of the materialising kernel on the stride-8 PAF (bit-identical to
        // reading the materialised paf_mat[y][x], tests/test_gpu_parity.py: lean == materialised): the stride-8 planes
        // are L2-resident, while gathers from the 36 MB-per-image paf_mat go to DRAM.
        src.ptr = a.paf; src.mode = PAF_LO_BILINEAR;
    } else {
        RefParams p;
        p.heat = a.heat; p.n = a.n; p.h = a.h; p.w = a.w; p.layout = a.layout; p.thr = a.thr;
        p.raw = c->raw; p.raw_count = c->raw_count; p.raw_cap = c->max_peaks; p.cubic = c->cubic;
        p.gauss = c->gauss;
        p.refine = a.frontend == EKP_FRONTEND_REFERENCE ? 1 : (a.frontend == EKP_FRONTEND_REFERENCE_GAUSS ? 2 : 0);
        CU(launch_ref_frontend(p, st));
        c->launches += ref_frontend_launches(p.refine);
        if (a.paf_mat) { CU(launch_upsample_nearest(a.paf, a.layout, a.n, a.h, a.w, EKP_PAF_CH, a.paf_mat, st)); c->launches += 1; }
        if (a.heat_mat) { CU(launch_upsample_nearest(a.heat, a.layout, a.n, a.h, a.w, EKP_HEAT_CH, a.heat_mat, st)); c->launches += 1; }
        src.ptr = a.paf; src.mode = PAF_LO_NEAREST;  // == paf_mat[y][x] exactly (cv2 INTER_NEAREST x8)
    }
    return run_back_half(c, a.n, /*id_from_key=*/0, src, /*h1=*/8 * a.h, st);
}

static bool same_args(const PostArgs& a, const PostArgs& b) {
    return a.heat == b.heat && a.paf == b.paf && a.heat_host == b.heat_host && a.paf_host == b.paf_host && a.heat16 == b.heat16 &&
           a.paf16 == b.paf16 && a.dtype == b.dtype && a.n == b.n && a.h == b.h &&
           a.w == b.w && a.layout == b.layout && a.frontend == b.frontend && memcmp(&a.thr, &b.thr, sizeof(float)) == 0 &&
           a.heat_mat == b.heat_mat && a.paf_mat == b.paf_mat;
}

// A context keeps the graphs of its last kMaxGraphs keys, the least recently used one evicted first: a stream of frames
// through the same buffers replays one, and a few shapes or buffer sets in turn each keep theirs.
static const size_t kMaxGraphs = 8;

int launch_cached(ekp_ctx* c, const GraphKey& key, unsigned long long host_epoch, cudaStream_t st,
                  const std::function<int(cudaStream_t)>& enqueue) {
    static const bool graphs_off = getenv("EKP_GRAPHS") && atoi(getenv("EKP_GRAPHS")) == 0;
    if (graphs_off || c->timing || !c->graphs_ok) return enqueue(st);
    std::vector<GraphEntry>& G = c->graphs;
    GraphEntry* hit = nullptr;
    for (size_t i = 0; i < G.size(); i++) {
        if (!same_args(G[i].key.batch, key.batch) || memcmp(G[i].key.scene, key.scene, sizeof(key.scene)) != 0) continue;
        if (G[i].host_epoch == host_epoch) { hit = &G[i]; break; }
        cudaGraphExecDestroy(G[i].exec);  // captured before a host block was released: capture again
        G.erase(G.begin() + (long) i);
        break;
    }
    if (!hit) {
        if (!c->cap_stream) CU(cudaStreamCreateWithFlags(&c->cap_stream, cudaStreamNonBlocking));
        const long long before = c->launches;
        cudaGraph_t graph = nullptr;
        CU(cudaStreamBeginCapture(c->cap_stream, cudaStreamCaptureModeThreadLocal));
        int rc = enqueue(c->cap_stream);
        cudaError_t ce = cudaStreamEndCapture(c->cap_stream, &graph);
        const int kernels = (int) (c->launches - before);
        c->launches = before;  // counted when the graph is launched
        cudaGraphExec_t exec = nullptr;
        if (rc == EKP_OK && ce == cudaSuccess && graph) ce = cudaGraphInstantiate(&exec, graph, 0);
        if (graph) cudaGraphDestroy(graph);
        if (rc != EKP_OK || ce != cudaSuccess || !exec) {  // no graph on this driver / for this sequence: stay eager from now on
            cudaGetLastError();
            c->graphs_ok = false;
            return enqueue(st);
        }
        if (G.size() >= kMaxGraphs) {  // evict the least recently used
            size_t lru = 0;
            for (size_t i = 1; i < G.size(); i++) if (G[i].stamp < G[lru].stamp) lru = i;
            cudaGraphExecDestroy(G[lru].exec);
            G.erase(G.begin() + (long) lru);
        }
        G.push_back(GraphEntry{key, exec, kernels, 0, host_epoch});
        hit = &G.back();
    }
    hit->stamp = ++c->graph_clock;
    CU(cudaGraphLaunch(hit->exec, st));
    c->launches += hit->kernels;
    c->graph_launches += 1;
    return EKP_OK;
}

static int submit_batch(ekp_ctx* c, const PostArgs& a, cudaStream_t st) {
    if (c->has_run && c->last_stream != st) CU(cudaStreamWaitEvent(st, c->done, 0));  // the work buffers are per context
    if (a.frontend == EKP_FRONTEND_DENSE) {
        int rc = ensure_tables(c, a.h, a.w, st);
        if (rc) return rc;
    }
    GraphKey key = {};
    key.batch = a;
    const unsigned long long epoch = a.heat_host ? g_host_frees.load(std::memory_order_acquire) : 0;
    int rc = launch_cached(c, key, epoch, st, [&](cudaStream_t q) { return enqueue_batch(c, a, q); });
    if (rc) return rc;
    c->map_h = 8 * a.h; c->map_w = 8 * a.w;
    return finish_submit(c, a.n, st);
}

// the context's float32 input block [heat | paf] (host entry: the copy target; 16-bit inputs: the widening target)
static int ensure_in_block(ekp_ctx* c) {
    if (!c->in_block)  // ONE staging block: heat, directly followed by paf (so adjacent host tensors arrive with one copy)
        CU(cudaMalloc((void**) &c->in_block, sizeof(float) * (size_t) c->max_batch * c->max_h * c->max_w * (EKP_HEAT_CH + EKP_PAF_CH)));
    return EKP_OK;
}

// the checks and batch arguments postprocess_dev and postprocess_host have in common
static int post_args(const ekp_ctx* c, const void* heat, const void* paf, int dtype, int n, int h, int w, int layout, float thr_heat,
                     int frontend, const char* who, PostArgs* a) {
    int rc = check_shape(c, n, h, w, layout, who);
    if (rc) return rc;
    if (frontend != EKP_FRONTEND_DENSE && frontend != EKP_FRONTEND_REFERENCE && frontend != EKP_FRONTEND_REFERENCE_COARSE &&
        frontend != EKP_FRONTEND_REFERENCE_GAUSS)
        return fail(EKP_ERR_ARG, "%s: frontend %d", who, frontend);
    if (!heat || !paf) return fail(EKP_ERR_ARG, "%s: NULL input", who);
    if (dtype != EKP_DTYPE_F32 && dtype != EKP_DTYPE_BF16 && dtype != EKP_DTYPE_F16)
        return fail(EKP_ERR_ARG, "%s: dtype %d (EKP_DTYPE_F32 0, EKP_DTYPE_BF16 1, EKP_DTYPE_F16 2)", who, dtype);
    if (dtype != EKP_DTYPE_F32 && ((reinterpret_cast<uintptr_t>(heat) | reinterpret_cast<uintptr_t>(paf)) & 1u))
        return fail(EKP_ERR_ARG, "%s: 16-bit heat / paf must be 2-byte aligned", who);
    *a = PostArgs{};
    a->dtype = dtype; a->n = n; a->h = h; a->w = w; a->layout = layout; a->frontend = frontend; a->thr = thr_heat;
    return EKP_OK;
}

static int postprocess_dev(ekp_ctx* c, const void* heat, const void* paf, int dtype, int n, int h, int w, int layout, float thr_heat,
                           int frontend, float* heat_mat, float* paf_mat, void* stream, const char* who) {
    PostArgs a;
    int rc = post_args(c, heat, paf, dtype, n, h, w, layout, thr_heat, frontend, who, &a);
    if (rc) return rc;
    if (heat_mat && !paf_mat) return fail(EKP_ERR_ARG, "%s: heat_mat without paf_mat", who);
    if ((reinterpret_cast<uintptr_t>(heat_mat) | reinterpret_cast<uintptr_t>(paf_mat)) & 15u)
        return fail(EKP_ERR_ARG, "%s: heat_mat / paf_mat must be 16-byte aligned (they are written with 16-byte bulk copies)", who);
    if (dtype == EKP_DTYPE_F32 && ((reinterpret_cast<uintptr_t>(heat) | reinterpret_cast<uintptr_t>(paf)) & 3u))
        return fail(EKP_ERR_ARG, "%s: heat / paf must be 4-byte aligned", who);
    CU(cudaSetDevice(c->device));
    if (dtype == EKP_DTYPE_F32) {
        a.heat = static_cast<const float*>(heat); a.paf = static_cast<const float*>(paf);
    } else {
        rc = ensure_in_block(c);
        if (rc) return rc;
        a.heat16 = heat; a.paf16 = paf;
        a.heat = c->in_block; a.paf = c->in_block + (size_t) n * h * w * EKP_HEAT_CH;
    }
    a.heat_mat = heat_mat; a.paf_mat = paf_mat;
    return submit_batch(c, a, (cudaStream_t) stream);
}

static int postprocess_host(ekp_ctx* c, const void* heat_host, const void* paf_host, int dtype, int n, int h, int w, int layout,
                            float thr_heat, int frontend, int materialize, void* stream, const char* who) {
    PostArgs a;
    int rc = post_args(c, heat_host, paf_host, dtype, n, h, w, layout, thr_heat, frontend, who, &a);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t) stream;
    CU(cudaSetDevice(c->device));
    rc = ensure_in_block(c);
    if (rc) return rc;
    if (dtype != EKP_DTYPE_F32 && !c->in_block16)  // the 16-bit copy target, laid out like in_block
        CU(cudaMalloc(&c->in_block16, 2 * (size_t) c->max_batch * c->max_h * c->max_w * (EKP_HEAT_CH + EKP_PAF_CH)));
    const size_t hw = (size_t) h * w;
    if (materialize) {
        const size_t heat_n = (size_t) n * hw * 64 * EKP_HEAT_CH, paf_n = (size_t) n * hw * 64 * EKP_PAF_CH;
        if (c->mat_heat_cap < heat_n || c->mat_paf_cap < paf_n) {
            rc = quiesce(c, st);  // the old tensors
            if (rc == EKP_OK) rc = grow(c->mat_heat, c->mat_heat_cap, heat_n);
            if (rc == EKP_OK) rc = grow(c->mat_paf, c->mat_paf_cap, paf_n);
            if (rc) return rc;
        }
        a.heat_mat = c->mat_heat; a.paf_mat = c->mat_paf;
    }
    const size_t elem = dtype == EKP_DTYPE_F32 ? sizeof(float) : 2;
    a.heat_host = heat_host; a.paf_host = paf_host;
    a.h2d_heat_bytes = elem * (size_t) n * hw * EKP_HEAT_CH;
    a.h2d_paf_bytes = elem * (size_t) n * hw * EKP_PAF_CH;
    a.heat = c->in_block; a.paf = c->in_block + (size_t) n * hw * EKP_HEAT_CH;
    if (dtype != EKP_DTYPE_F32) { a.heat16 = c->in_block16; a.paf16 = static_cast<char*>(c->in_block16) + a.h2d_heat_bytes; }
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
    int rc = run_back_half(c, n, /*id_from_key=*/1, paf_source(PAF_FULL_HWC, paf_mat, nullptr, H, W, C), h1, st);
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

// ---- readers of the last run's records on the device (draw.cu, results_device.cu) ----------------------------------
// Puts what enqueue() issues on `st` after the last run (and after earlier readers: the draw's keys), and the context's
// next run on any stream after it, so that run cannot overwrite the records while they are read (submit_batch waits for
// `done`).  No host wait.
static int after_run(ekp_ctx* c, cudaStream_t st, const std::function<int()>& enqueue) {
    CU(cudaSetDevice(c->device));
    if (c->last_stream != st) CU(cudaStreamWaitEvent(st, c->done, 0));
    int rc = enqueue();
    if (rc) return rc;
    CU(cudaEventRecord(c->done, st));
    c->last_stream = st;
    return EKP_OK;
}

extern "C" int ekp_draw_humans(ekp_ctx* c, unsigned char* frames, int n, int H, int W, void* stream) {
    if (!c) return fail(EKP_ERR_ARG, "ekp_draw_humans: NULL context");
    if (!c->has_run) return fail(EKP_ERR_STATE, "ekp_draw_humans: no run has been submitted on this context");
    if (!frames) return fail(EKP_ERR_ARG, "ekp_draw_humans: NULL frames");
    if (n != c->last_n) return fail(EKP_ERR_ARG, "ekp_draw_humans: %d frames for a run of %d images", n, c->last_n);
    if (H < 1 || W < 1 || H > EKP_DRAW_MAX_SIDE || W > EKP_DRAW_MAX_SIDE)
        return fail(EKP_ERR_ARG, "ekp_draw_humans: frame %dx%d outside [1x1, %dx%d]", H, W, EKP_DRAW_MAX_SIDE, EKP_DRAW_MAX_SIDE);
    cudaStream_t st = (cudaStream_t) stream;
    return after_run(c, st, [&]() {
        const size_t pixels = (size_t) n * H * W;
        if (c->draw_keys_cap < pixels) {
            CU(cudaEventSynchronize(c->done));  // no draw in flight may still use the old keys
            int rc = grow(c->draw_keys, c->draw_keys_cap, pixels);
            if (rc) return rc;
            c->draw_epoch = 0xffff;  // cleared below
        }
        if (c->draw_epoch == 0xffff) {  // the epoch would wrap: keys of old draws could equal or exceed this draw's
            CU(cudaMemsetAsync(c->draw_keys, 0, sizeof(unsigned) * c->draw_keys_cap, st));
            c->draw_epoch = 0;
        }
        c->draw_epoch += 1;
        CU(launch_draw(c->last_records, c->lay, c->max_humans, c->map_h, c->map_w, frames, n, H, W, c->draw_keys, c->draw_epoch, st));
        c->launches += 2;
        return (int) EKP_OK;
    });
}

extern "C" int ekp_results_device(ekp_ctx* c, int n, const ekp_device_results* out, void* stream) {
    if (!c || !out) return fail(EKP_ERR_ARG, "ekp_results_device: NULL %s", c ? "out" : "context");
    if (!c->has_run) return fail(EKP_ERR_STATE, "ekp_results_device: no run has been submitted on this context");
    if (n != c->last_n) return fail(EKP_ERR_ARG, "ekp_results_device: tables for %d images, the run had %d", n, c->last_n);
    const void* ptrs[] = {out->num_humans, out->overflow, out->n_peaks, out->subset, out->parts, out->scores};
    bool any = false;
    for (const void* p : ptrs) {
        if (reinterpret_cast<uintptr_t>(p) & 3u) return fail(EKP_ERR_ARG, "ekp_results_device: a pointer is not 4-byte aligned");
        any = any || p;
    }
    if (!any) return EKP_OK;
    cudaStream_t st = (cudaStream_t) stream;
    return after_run(c, st, [&]() {
        CU(launch_results_export(c->last_records, c->lay, c->max_humans, n, *out, st));
        c->launches += 1;
        return (int) EKP_OK;
    });
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
        CU(cudaStreamSynchronize(st));  // no kernel in flight may still read the old tables
        c->prep_sh = c->prep_sw = 0;
        rc = grow(c->prep_tab, c->prep_tab_cap, tab_bytes);
        if (rc) return rc;
        CU(cudaMemcpy(c->prep_tab, ofs.data(), sizeof(int) * ofs.size(), cudaMemcpyHostToDevice));
        CU(cudaMemcpy(c->prep_tab + sizeof(int) * ofs.size(), coef.data(), sizeof(short) * coef.size(), cudaMemcpyHostToDevice));
        c->prep_sh = sh; c->prep_sw = sw; c->prep_dest = dest_size; c->prep_rh = rh; c->prep_rw = rw;
    }
    const int* xofs = (const int*) c->prep_tab;
    const int* yofs = xofs + rw;
    const short* ialpha = (const short*) (c->prep_tab + sizeof(int) * ((size_t) rw + rh));
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
    DenseParams p = dense_params(c, heat, n, h, w, layout);
    p.thr = INFINITY; p.smooth_out = smooth_out;
    CU(launch_dense_frontend(p, st));
    c->launches += 1;
    return EKP_OK;
}
