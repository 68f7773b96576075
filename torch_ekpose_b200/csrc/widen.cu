// widen.cu -- 16-bit network outputs (bf16 / fp16 heat and PAF maps, e.g. from torch.autocast) widened to float32 on
// the device, element for element in the caller's layout, into the context's float32 input block.  The front-end and
// stage 4-5 kernels then run unchanged on that block, so a 16-bit batch gives exactly what the float32 path gives on
// x.float(): bf16 -> f32 and fp16 -> f32 are exact (finite values, +-0, subnormals, +-inf; a NaN stays a NaN).
//
// One launch covers both tensors.  Each is a segment: a scalar head up to the first 16-byte-aligned source element, a
// body of 8-element groups (one 16-byte load, two 16-byte stores when the destination is 16-byte aligned at the group,
// else eight 4-byte stores), a scalar tail.  The front-end re-reads the block right after this kernel (36 MB at
// 64 x 46x54, inside the 126 MB L2), so the stores keep the default cache policy.
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <string.h>

#include <algorithm>

#include "common.cuh"

namespace ekp {

struct WidenSeg {
    const unsigned short* src;  // 2-byte aligned
    float* dst;                 // 4-byte aligned
    size_t n;                   // elements
    unsigned head;              // scalar elements before the first 16-byte-aligned source element (<= 7)
    size_t groups;              // 8-element groups of the body
    bool dst_vec;               // dst + head is 16-byte aligned (then every group's destination is)
};

template <int DT>
__device__ __forceinline__ float widen1(unsigned short v) {
    if (DT == EKP_DTYPE_BF16) return __uint_as_float((unsigned) v << 16);
    return __half2float(__ushort_as_half(v));
}

template <int DT>
__device__ __forceinline__ float2 widen2(unsigned w) {  // two packed 16-bit values, the lower one first in memory
    if (DT == EKP_DTYPE_BF16) return make_float2(__uint_as_float(w << 16), __uint_as_float(w & 0xffff0000u));
    __half2 h;
    memcpy(&h, &w, sizeof(h));
    return __half22float2(h);
}

template <int DT>
__device__ __forceinline__ void widen_group(const WidenSeg& s, size_t g) {
    const size_t e = s.head + 8 * g;
    const uint4 v = __ldg(reinterpret_cast<const uint4*>(s.src + e));
    const float2 a = widen2<DT>(v.x), b = widen2<DT>(v.y), c = widen2<DT>(v.z), d = widen2<DT>(v.w);
    float* o = s.dst + e;
    if (s.dst_vec) {
        reinterpret_cast<float4*>(o)[0] = make_float4(a.x, a.y, b.x, b.y);
        reinterpret_cast<float4*>(o)[1] = make_float4(c.x, c.y, d.x, d.y);
    } else {
        o[0] = a.x; o[1] = a.y; o[2] = b.x; o[3] = b.y; o[4] = c.x; o[5] = c.y; o[6] = d.x; o[7] = d.y;
    }
}

template <int DT>
__global__ void __launch_bounds__(256) widen_kernel(const WidenSeg s0, const WidenSeg s1) {
    const size_t stride = (size_t) gridDim.x * blockDim.x;
    const size_t t0 = (size_t) blockIdx.x * blockDim.x + threadIdx.x;
    for (size_t g = t0; g < s0.groups; g += stride) widen_group<DT>(s0, g);
    for (size_t g = t0; g < s1.groups; g += stride) widen_group<DT>(s1, g);
    if (blockIdx.x == 0 && threadIdx.x < 32) {  // heads (j < 8) and tails (j >= 8) of both segments, one element each
        const WidenSeg& s = threadIdx.x < 16 ? s0 : s1;
        const unsigned j = threadIdx.x & 15u;
        const size_t tail0 = s.head + 8 * s.groups;
        const size_t e = j < 8 ? (size_t) j : tail0 + (j - 8);
        if ((j < 8 && j < s.head) || (j >= 8 && e < s.n)) s.dst[e] = widen1<DT>(s.src[e]);
    }
}

static WidenSeg make_seg(const void* src, float* dst, size_t n) {
    WidenSeg s;
    s.src = static_cast<const unsigned short*>(src);
    s.dst = dst;
    s.n = n;
    const unsigned mis = (unsigned) (reinterpret_cast<uintptr_t>(src) & 15u);  // even: the caller checked 2-byte alignment
    s.head = (unsigned) std::min<size_t>(n, ((16u - mis) & 15u) / 2u);
    s.groups = (n - s.head) / 8;
    s.dst_vec = ((reinterpret_cast<uintptr_t>(dst + s.head)) & 15u) == 0;
    return s;
}

// heat16 [n_heat] and paf16 [n_paf] 16-bit elements of type `dtype` (EKP_DTYPE_BF16 / EKP_DTYPE_F16) -> float32 at
// heat / paf.  One kernel launch.
cudaError_t launch_widen(const void* heat16, const void* paf16, size_t n_heat, size_t n_paf, int dtype, float* heat, float* paf,
                         cudaStream_t stream) {
    const WidenSeg s0 = make_seg(heat16, heat, n_heat), s1 = make_seg(paf16, paf, n_paf);
    int dev = 0, sms = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess) return e;
    const size_t groups = s0.groups + s1.groups;
    const size_t want = (groups + 255) / 256;
    const int blocks = (int) std::max<size_t>(1, std::min<size_t>(want, (size_t) sms * 8));  // 8 x 256 threads fill an SM
    if (dtype == EKP_DTYPE_BF16) widen_kernel<EKP_DTYPE_BF16><<<blocks, 256, 0, stream>>>(s0, s1);
    else widen_kernel<EKP_DTYPE_F16><<<blocks, 256, 0, stream>>>(s0, s1);
    return cudaGetLastError();
}

}  // namespace ekp
