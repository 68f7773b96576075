// common.cuh -- shared device-side types for libekpose_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/ekpose_b200.h"

namespace ekp {

// Unordered peak record produced by stages 1-3 (or by the peak-list ingest of process_paf).
// Ordering is restored by peaks_sort_kernel from (part, key): the reference emits peaks in
// (part, y, x) order (paf_to_pose.py:36, :350-352) and process_paf buckets by part keeping input
// order (pafprocess.cpp:24-43).
struct RawPeak {
    int x;          // full-resolution column
    int y;          // full-resolution row
    float score;
    int part;       // 0..17
    unsigned key;   // order within the part: (row << 16 | col) of the maximum, or the input index
};

struct __align__(16) Conn {  // pafprocess.h:45-51, plus the two score sums the assembly forms from it
    int cid1, cid2;
    float score;
    float s_ext;   // peak_score(cid2) + score                      (pafprocess.cpp:150/171: a row is extended by part2)
    float s_new;   // (peak_score(cid1) + peak_score(cid2)) + score (:179-181: a new row), peak scores looked up by
                   // cid in the part-sorted table like the reference's peak_infos_line[cid]
    int pad0, pad1, pad2;
};

// how stage 4 obtains paf_mat[y][x][ch]
enum PafMode {
    PAF_FULL_HWC = 0,      // gather from a materialised full-resolution [H][W][C] tensor
    PAF_LO_NEAREST = 1,    // paf_lo[y>>3][x>>3]   (== cv2 INTER_NEAREST x8, paf_to_pose.py:356-357)
    PAF_LO_BILINEAR = 2,   // bilinear x8 of paf_lo, same arithmetic as the materialising kernel
    PAF_PACKED = 3         // the samples themselves, gathered beforehand: float2 [(pair_base[limb] + pair) * 10 + i]
                           // (host-pointer process_paf: only the values stage 4 reads are uploaded)
};

struct PafSource {
    const float* ptr;  // full-res HWC tensor, or stride-8 tensor
    int mode;
    int layout;        // of the stride-8 tensor (EKP_LAYOUT_*)
    int H, W, C;       // full-resolution dims and channel count
    int h, w;          // stride-8 dims (modes 1, 2)
    const int* pair_base;  // [20] prefix of nA*nB over the limbs (mode 3)
    int ids_are_rows;      // 1: a peak's id IS its row in the part-sorted table (front-end paths), so the score the
                           // reference looks up as peak_infos_line[cid] is the peak's own; 0: process_paf input order
};

// pafprocess.h:16-24
__constant__ const int kPairsNet[EKP_NUM_LIMB][2] = {
    {12, 13}, {20, 21}, {14, 15}, {16, 17}, {22, 23}, {24, 25}, {0, 1},   {2, 3},   {4, 5},   {6, 7},
    {8, 9},   {10, 11}, {28, 29}, {30, 31}, {34, 35}, {32, 33}, {36, 37}, {18, 19}, {26, 27}};
__constant__ const int kPairs[EKP_NUM_LIMB][2] = {
    {1, 2},   {1, 5},   {2, 3},  {3, 4},   {5, 6},   {6, 7},  {1, 8},   {8, 9},  {9, 10}, {1, 11},
    {11, 12}, {12, 13}, {1, 0},  {0, 14},  {14, 16}, {0, 15}, {15, 17}, {2, 16}, {5, 17}};

// bilinear x8 with half-pixel centres: source index pair and weight for full-res coordinate D.
// s = (D + 0.5)/8 - 0.5;  i0 = floor(s) = (D+4)/8 - 1;  t = s - i0 = (2*((D+4)%8) + 1)/16 (exact).
__device__ __forceinline__ void bilin_coord(int D, int n, int& i0, int& i1, float& t) {
    const int q = D + 4;
    i0 = (q >> 3) - 1;
    t = (float) (2 * (q & 7) + 1) * 0.0625f;
    i1 = min(i0 + 1, n - 1);
    i0 = max(i0, 0);
}
// a + t*(b - a) with one rounding in the subtract and one in the fused multiply-add; the CPU
// oracle uses fmaf() for the same expression.
__device__ __forceinline__ float lerp1(float a, float b, float t) { return fmaf(t, __fsub_rn(b, a), a); }

__device__ __forceinline__ float lo_at(const float* lo, int layout, int img, int C, int h, int w, int c, int j, int i) {
    return layout == EKP_LAYOUT_NCHW ? __ldg(lo + (((size_t) img * C + c) * h + j) * w + i)
                                     : __ldg(lo + (((size_t) img * h + j) * w + i) * C + c);
}

// ---- TMA bulk load of a contiguous, 16-byte aligned range into shared memory (cp.async.bulk global -> shared, SASS
// UBLKCP.S.G), completion counted in bytes on an mbarrier: one thread arms the barrier and issues the copy, every
// thread waits on the barrier's phase.
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((unsigned) __cvta_generic_to_shared(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"((unsigned) __cvta_generic_to_shared(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_load(void* sdst, const void* gsrc, unsigned bytes, unsigned long long* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     (unsigned) __cvta_generic_to_shared(sdst)),
                 "l"(gsrc), "r"(bytes), "r"((unsigned) __cvta_generic_to_shared(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"((unsigned) __cvta_generic_to_shared(bar)),
        "r"(parity)
        : "memory");
}

// One packed result record per image, so a batch's results are a single device-to-host copy:
//   [0]           int num_humans, int n_peaks, unsigned overflow, int pad
//   [off_subset]  float  subset[max_humans][20]      rows as the reference keeps them
//   [off_hparts]  ekp_peak parts[max_humans][18]     (x, y, score, cid or -1) per human and part
//   [off_hscore]  float  score[max_humans]           subset[18] / subset[19]
struct ResultLayout {
    size_t stride, off_subset, off_hparts, off_hscore;
};

// cudaFuncAttributeMaxDynamicSharedMemorySize is per kernel and device, shared by every context: a context with
// smaller capacities must never LOWER it under a bigger one.  Raises the limit to `bytes` if it is below.
template <typename Kernel>
inline cudaError_t raise_dynamic_smem_limit(Kernel kernel, size_t bytes) {
    cudaFuncAttributes attr;
    cudaError_t e = cudaFuncGetAttributes(&attr, kernel);
    if (e != cudaSuccess) return e;
    if ((size_t) attr.maxDynamicSharedSizeBytes >= bytes) return cudaSuccess;
    return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) bytes);
}

// pycocotools' keypoint variances: sigmas = array([...]) / 10.0, vars = (sigmas * 2) ** 2, in float64 (on the host,
// into the kernels' arguments).  One copy for the tracker's similarity (track.cu) and the COCO evaluation (coco_eval.cu).
inline void oks_vars(double var[17]) {
    const double s[17] = {.26, .25, .25, .35, .35, .79, .79, .72, .72, .62, .62, 1.07, 1.07, .87, .87, .89, .89};
    for (int j = 0; j < 17; j++) {
        const double sg = s[j] / 10.0;
        var[j] = (sg * 2) * (sg * 2);
    }
}

// The track-table rules of a sequence of frames, one copy for the tracker (track.cu) and the smoother (smooth.cu): an
// entry last seen at frame last_seen is dropped at frame last_seen + max_age + 2, and a new entry that finds no free one
// takes that of the smallest (last_seen, id) among those not seen in the current frame.
__host__ __device__ __forceinline__ bool expired(int last_seen, int f, int max_age) {
    return (long long) f - last_seen > (long long) max_age + 1;
}
__host__ __device__ __forceinline__ bool evict_first(int seen_a, int id_a, int seen_b, int id_b) {
    return seen_a < seen_b || (seen_a == seen_b && id_a < id_b);
}

// launch parameter blocks --------------------------------------------------------------------
struct AsmParams {
    const ekp_peak* line;      // [n][max_peaks] part-sorted peak table
    int max_peaks;
    const int* n_peaks;        // [n]
    const int* part_off;       // [n][20] ([19] = number of raw peaks, the bound of every id)
    const Conn* conns;         // [n][19][max_part]
    const int* n_conns;        // [n][19]
    int max_part, max_humans;
    int conn_cap;              // staged connection records per image (set by launch_assemble)
    const unsigned* overflow;  // [n]
    unsigned char* records;    // [n] packed result records
    ResultLayout lay;
};

struct ConnectParams {
    const ekp_peak* line;
    const int* part_off;
    int max_peaks, max_part, max_cand;
    PafSource paf;
    int h1;
    int by_sample_max_pairs;   // a block scores with ten lanes per pair when it has at most this many pairs (else one thread per pair)
    Conn* conns;               // [n][19][max_part]
    int* n_conns;              // [n][19]
    unsigned* overflow;
};

struct DenseParams {
    const float* heat;
    const float* paf;
    int n, h, w, layout;
    float thr;
    const float* ax;   // [8w][8] polyphase taps along x (5 used)
    const float* ay;   // [8h][8] along y
    float* heat_mat;   // nullable
    float* paf_mat;    // nullable
    float* smooth_out; // nullable debug output [n][8h][8w][18]
    RawPeak* raw;
    int* raw_count;
    int raw_cap;
    int tile_wl;       // stride-8 columns per tile
};

struct RefParams {
    const float* heat;
    int n, h, w, layout;
    float thr;
    RawPeak* raw;
    int* raw_count;
    int raw_cap;
    const float* cubic; // [8][4] cv2 bicubic coefficients for t = (2k+1)/16
    const double* gauss; // [13] scipy gaussian_filter(sigma=3) weights w[-12] .. w[0] (refine == 2)
    int refine;         // 0: report the stride-8 maxima themselves (NMS(bool_refine_center=False), paf_to_pose.py:119-122);
                        // 1: bicubic refinement; 2: ... with the Gaussian on the upsampled patch (bool_gaussian_filt, :111-112)
};

}  // namespace ekp
