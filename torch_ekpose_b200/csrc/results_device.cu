// results_device.cu -- the last run's result tables written into caller-owned DEVICE buffers (ekp_results_device, and
// ekp_results_device_peaks for the peak table): the device counterpart of ekp_results / ekp_results_humans /
// ekp_results_parts, ordered on a stream after the run, with no host wait.
//
// Each image's packed record (ResultLayout) holds the header, then the subset rows, the per-human part table and the
// human scores, every region starting on a 16-byte boundary.  Rows below min(num_humans, max_humans) are copied byte for
// byte; every row from there up to max_humans is written as zero bytes, which is what the host readers hand back there
// (they fill arrays that start out zeroed), so a copied-back table equals the host one padding included, whatever the
// destination held before.  A region moves in 16-byte units when its destination is 16-byte aligned for every image,
// else in 4-byte units.  A few MB per batch: the kernel is latency-bound, so the grid spreads each image over a few
// blocks rather than looping long in one.
#include "common.cuh"

namespace ekp {

struct ExportRegion {
    unsigned* dst;     // [n][max_humans * row_words], or nullptr (not written)
    unsigned src_off;  // byte offset of the region in a record (16-byte aligned)
    int row_words;     // 4-byte words per row
    bool vec;          // dst is 16-byte aligned for every image (and row_words * max_humans % 4 == 0)
};

struct ExportParams {
    const unsigned char* records;
    size_t stride;
    int max_humans;
    int* num_humans;
    unsigned* overflow;
    int* n_peaks;
    ExportRegion reg[3];  // subset, parts, scores
};

// words [0, valid) of src to dst and zeros to [valid, total), units first, first + step, ... of this image
__device__ __forceinline__ void copy_region(const unsigned* src, unsigned* dst, int valid, int total, bool vec, int first, int step) {
    if (vec) {
        for (int q = first; 4 * q < total; q += step) {
            uint4 v = make_uint4(0u, 0u, 0u, 0u);
            if (4 * q < valid) {
                v = reinterpret_cast<const uint4*>(src)[q];
                const int k = valid - 4 * q;  // words of this unit below `valid`; only the scores' rows are not whole units
                if (k < 2) v.y = 0u;
                if (k < 3) v.z = 0u;
                if (k < 4) v.w = 0u;
            }
            reinterpret_cast<uint4*>(dst)[q] = v;
        }
    } else {
        for (int w = first; w < total; w += step) dst[w] = w < valid ? src[w] : 0u;
    }
}

// grid (chunks, n): blocks blockIdx.x of image blockIdx.y share its regions in a block-strided loop
__global__ void __launch_bounds__(256) results_export_kernel(const ExportParams P) {
    const int img = blockIdx.y;
    const unsigned char* rec = P.records + P.stride * (size_t) img;
    const int4 head = *reinterpret_cast<const int4*>(rec);  // num_humans, n_peaks, overflow, pad
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        if (P.num_humans) P.num_humans[img] = head.x;
        if (P.n_peaks) P.n_peaks[img] = head.y;
        if (P.overflow) P.overflow[img] = (unsigned) head.z;
    }
    const int rows = min(head.x, P.max_humans);
    const int first = blockIdx.x * blockDim.x + threadIdx.x, step = gridDim.x * blockDim.x;
#pragma unroll
    for (int r = 0; r < 3; r++) {
        const ExportRegion& g = P.reg[r];
        if (!g.dst) continue;
        const int total = P.max_humans * g.row_words;
        copy_region(reinterpret_cast<const unsigned*>(rec + g.src_off), g.dst + (size_t) img * total, rows * g.row_words, total, g.vec,
                    first, step);
    }
}

cudaError_t launch_results_export(const unsigned char* records, const ResultLayout& lay, int max_humans, int n,
                                  const ekp_device_results& out, cudaStream_t stream) {
    ExportParams P;
    P.records = records; P.stride = lay.stride; P.max_humans = max_humans;
    P.num_humans = out.num_humans; P.overflow = out.overflow; P.n_peaks = out.n_peaks;
    void* dst[3] = {out.subset, out.parts, out.scores};
    const size_t off[3] = {lay.off_subset, lay.off_hparts, lay.off_hscore};
    const int words[3] = {EKP_SUBSET_COLS, EKP_NUM_PART * 4, 1};
    int units = 1;  // of the largest region of one image: what the grid's x extent is sized for
    for (int r = 0; r < 3; r++) {
        const int total = max_humans * words[r];
        P.reg[r].dst = static_cast<unsigned*>(dst[r]);
        P.reg[r].src_off = (unsigned) off[r];
        P.reg[r].row_words = words[r];
        P.reg[r].vec = (reinterpret_cast<uintptr_t>(dst[r]) & 15u) == 0 && total % 4 == 0;
        if (dst[r]) units = max(units, P.reg[r].vec ? total / 4 : total);
    }
    const int kThreads = 256, kUnitsPerThread = 2;
    const unsigned chunks = (unsigned) ((units + kThreads * kUnitsPerThread - 1) / (kThreads * kUnitsPerThread));
    results_export_kernel<<<dim3(chunks, (unsigned) n), kThreads, 0, stream>>>(P);
    return cudaGetLastError();
}

// ---- the peak table (ekp_results_device_peaks) -------------------------------------------------------------------------
// The context's part-sorted table line [n][max_peaks] and part_off [n][20] (the 20th entry is not exported), with each
// image's peak count taken from its record header as the host reader takes it.  Rows from min(n_peaks, max_peaks) on
// are written as zero bytes, like the people's padding above.
struct PeaksExportParams {
    const unsigned char* records;
    size_t stride;
    const unsigned* line;      // ekp_peak [n][max_peaks] as words
    const unsigned* part_off;  // [n][20]
    int max_peaks;
    int* n_peaks;
    unsigned* peaks;           // [n][max_peaks * 4] or nullptr
    int* part_off_out;         // [n][19] or nullptr
    bool vec;                  // peaks is 16-byte aligned (every image's table then is)
};

__global__ void __launch_bounds__(256) peaks_export_kernel(const PeaksExportParams P) {
    const int img = blockIdx.y;
    const int npk = reinterpret_cast<const int4*>(P.records + P.stride * (size_t) img)->y;  // num_humans, n_peaks, overflow, pad
    if (blockIdx.x == 0 && threadIdx.x == 0 && P.n_peaks) P.n_peaks[img] = npk;
    const int first = blockIdx.x * blockDim.x + threadIdx.x, step = gridDim.x * blockDim.x;
    const int total = 4 * P.max_peaks;
    if (P.peaks)
        copy_region(P.line + (size_t) img * total, P.peaks + (size_t) img * total, 4 * min(npk, P.max_peaks), total, P.vec, first, step);
    if (P.part_off_out)
        copy_region(P.part_off + (size_t) img * 20, reinterpret_cast<unsigned*>(P.part_off_out) + (size_t) img * 19, 19, 19, false,
                    first, step);
}

cudaError_t launch_peaks_export(const unsigned char* records, size_t stride, const ekp_peak* line, const int* part_off, int max_peaks,
                                int n, const ekp_device_peaks& out, cudaStream_t stream) {
    PeaksExportParams P;
    P.records = records; P.stride = stride; P.max_peaks = max_peaks;
    P.line = reinterpret_cast<const unsigned*>(line); P.part_off = reinterpret_cast<const unsigned*>(part_off);
    P.n_peaks = out.n_peaks; P.peaks = reinterpret_cast<unsigned*>(out.peaks); P.part_off_out = out.part_off;
    P.vec = (reinterpret_cast<uintptr_t>(out.peaks) & 15u) == 0;
    const int units = out.peaks ? (P.vec ? max_peaks : 4 * max_peaks) : 19;
    const int kThreads = 256, kUnitsPerThread = 2;
    const unsigned chunks = (unsigned) ((units + kThreads * kUnitsPerThread - 1) / (kThreads * kUnitsPerThread));
    peaks_export_kernel<<<dim3(chunks, (unsigned) n), kThreads, 0, stream>>>(P);
    return cudaGetLastError();
}

}  // namespace ekp
