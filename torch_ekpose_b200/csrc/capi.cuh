// capi.cuh -- internal to the host orchestration: capi.cu (the context API) and process_paf.cu (the reference operator
// surface).  The kernel sources do not include it.
#pragma once
#include <functional>
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
cudaError_t launch_results_export(const unsigned char* records, const ResultLayout& lay, int max_humans, int n,
                                  const ekp_device_results& out, cudaStream_t stream);
void debug_raster_host(int kind, int x0, int y0, int x1, int y1, int H, int W, unsigned char* mask);
void debug_draw_host(const int* num_humans, const ekp_peak* parts, int max_humans, int map_h, int map_w,
                     unsigned char* frames, int n, int H, int W);
}  // namespace ekp

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

// What a cached CUDA graph was captured for.  A batch of the context API is keyed by its arguments; process_paf's
// small-scene route by the shape and block size its launch arguments depend on.  Each leaves the other's fields zero.
struct GraphKey {
    PostArgs batch;
    long long scene[6];
};

// host_epoch: g_host_frees when a graph with host inputs was captured.  Its copy nodes refer to the pinned allocation that
// held them; once any block is released by ekp_host_free a new block may come back at the same address, so such graphs
// are not replayed across an ekp_host_free (they would copy from the released allocation).
struct GraphEntry { GraphKey key; cudaGraphExec_t exec; int kernels; unsigned long long stamp, host_epoch; };

struct ekp_ctx {
    int device = 0, max_batch = 0, max_h = 0, max_w = 0, max_peaks = 0, max_humans = 0;
    int max_part = EKP_MAX_PART, max_cand = EKP_MAX_CAND;  // peaks of one part / passing candidates of one limb, per image
    // device work buffers
    ekp::RawPeak* raw = nullptr;
    int* raw_count = nullptr;       // [max_batch]
    unsigned* overflow = nullptr;   // [max_batch]  (contiguous with raw_count: one memset)
    ekp_peak* line = nullptr;       // [max_batch][max_peaks]
    int* part_off = nullptr;        // [max_batch][20]
    int* n_peaks = nullptr;         // [max_batch]
    ekp::Conn* conns = nullptr;     // [max_batch][19][max_part]
    int* n_conns = nullptr;         // [max_batch][19]
    unsigned char* records = nullptr;  // [max_batch] packed result records (ResultLayout)
    const unsigned char* last_records = nullptr;  // where the last run's assembly wrote them (records, or pinned host)
    int map_h = 0, map_w = 0;       // the last run's full-resolution map, by which ekp_draw_humans normalises
    unsigned* draw_keys = nullptr;  // ekp_draw_humans' per-pixel keys (lazily, grown on demand)
    size_t draw_keys_cap = 0;       // pixels
    unsigned draw_epoch = 0;        // draws since the keys were last cleared (the high 16 bits of every key)
    ekp::ResultLayout lay = {};
    float* in_block = nullptr;      // staging for the host-buffer entry point: [heat | paf] of one batch, contiguous
                                    // (also where 16-bit inputs are widened to)
    void* in_block16 = nullptr;     // 16-bit [heat | paf] staging of the host-buffer entry point (lazily, half of in_block)
    float* mat_heat = nullptr;      // context-owned operator-surface tensors (host entry, lazily)
    float* mat_paf = nullptr;
    size_t mat_heat_cap = 0, mat_paf_cap = 0;
    float* ax = nullptr;            // dense taps for (tab_h, tab_w)
    float* ay = nullptr;
    int tab_h = 0, tab_w = 0;
    float* cubic = nullptr;         // [8][4]
    double* gauss = nullptr;        // [13]
    char* prep_tab = nullptr;       // resize tables of the input side for (prep_sh, prep_sw, prep_dest)
    size_t prep_tab_cap = 0;        // bytes
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
    // CUDA graphs of repeated submissions (launch_cached)
    std::vector<GraphEntry> graphs;
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

// The functions below are shared by the two host files only: they stay out of the library's dynamic symbol table.
#pragma GCC visibility push(hidden)

// ---- error reporting -------------------------------------------------------------------------
// Sets the message ekp_last_error() returns (per thread) and returns `code`.
int fail(int code, const char* fmt, ...);
#define CU(expr)                                                                                        \
    do {                                                                                                \
        cudaError_t _e = (expr);                                                                        \
        if (_e != cudaSuccess) return fail(EKP_ERR_CUDA, "%s: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)

// stages 4-5 + result copies, shared by every entry point; each adds the kernels it launches to c->launches
int run_peak_sort(ekp_ctx* c, int n, int id_from_key, cudaStream_t st);
// records_direct: device-visible pinned host memory the assembly writes the result records to itself (no D2H copy node)
int run_connect_assemble(ekp_ctx* c, int n, const ekp::PafSource& paf, int h1, cudaStream_t st, unsigned char* records_direct = nullptr);
// Stage 4's view of a caller's paf_mat [f1][f2][f3] (NHWC), in which a peak's id is its row in the caller's peak table: the
// tensor itself (PAF_FULL_HWC) or the samples gathered from it (PAF_PACKED, laid out by pair_base).
ekp::PafSource paf_source(int mode, const void* ptr, const int* pair_base, int f1, int f2, int f3);
// after a run has been put on `st` (eagerly or as a graph launch): results become readable when `done` fires
int finish_submit(ekp_ctx* c, int n, cudaStream_t st);

// Puts on `st` what enqueue(q) issues on a stream q, as a replay of the context's CUDA graph for `key`: captured and
// instantiated on the first use of the key, then one launch call instead of many stream operations, and no gaps
// between the small latency-bound kernels of stages 4-5.  host_epoch: see GraphEntry (0 without host inputs).
// Runs enqueue eagerly instead under EKP_GRAPHS=0, with per-stage timing, or once a capture has failed on this context.
int launch_cached(ekp_ctx* c, const GraphKey& key, unsigned long long host_epoch, cudaStream_t st,
                  const std::function<int(cudaStream_t)>& enqueue);
// Destroys the context's graphs: their nodes refer to buffers, so this goes with freeing any buffer they use.
void drop_graphs(ekp_ctx* c);

// Makes `p` hold at least `need` elements of T: device memory, or pinned host memory with GROW_PINNED.  A smaller buffer
// is freed, not copied, so the caller makes sure nothing in flight still uses it.  GROW_SLACK allocates half as much
// again, so that a slowly growing stream of scenes does not reallocate on every call.
enum { GROW_PINNED = 1, GROW_SLACK = 2 };
template <class T> int grow(T*& p, size_t& cap, size_t need, int flags = 0) {
    if (cap >= need) return EKP_OK;
    const bool pinned = flags & GROW_PINNED;
    if (p) { if (pinned) cudaFreeHost(p); else cudaFree(p); }
    p = nullptr; cap = 0;
    const size_t n = flags & GROW_SLACK ? need + need / 2 + 1024 : need;
    CU(pinned ? cudaMallocHost((void**) &p, sizeof(T) * n) : cudaMalloc((void**) &p, sizeof(T) * n));
    cap = n;
    return EKP_OK;
}

#pragma GCC visibility pop
