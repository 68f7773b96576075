// draw.cu -- the reference's draw_humans (lib/utils/common.py:252-275) on the device: the people of the last run painted
// onto n uint8 frames [n, H, W, 3], byte for byte what the reference's cv2 calls paint on the same people.
//
// Per image the people are a list of primitives in the reference's drawing order: human k of the table, its 18 part
// markers (cv2.circle(c, 3, colour, thickness=3)) in part order, then its 17 limbs (cv2.line(a, b, colour, 3)) in
// CocoPairsRender order; primitive s = 35 k + j.  Primitives overwrite each other, so a pixel ends up with the colour of
// the LAST primitive that covers it.  Each primitive is rasterised serially, by one thread, with a restatement of
// cv2's own integer arithmetic (drawing.cpp: ThickLine, FillConvexPoly, Line2, clipLine, Circle); the parallel part is
// only the order:
//   pass 1 (cover)  every primitive does atomicMax(key[pixel], tag(s)) on the pixels it paints;
//   pass 2 (paint)  one thread per 4 keys of the batch: a key of this draw names the last primitive s covering its
//                   pixel, and s names the colour (CocoColors[j], j = s mod 35 less 18 for a limb), written there.
// Frame pixels no primitive covers are neither read nor written.  tag(s) = epoch << 16 | (s + 1), the epoch counting
// the context's draws, so keys left by earlier draws are smaller than every key of this one and the key buffer needs no
// clearing between draws (only when the epoch wraps after 65535 draws).  Pass 2 scans the keys rather than
// rasterising every primitive again: a primitive's pixels are a serial walk, and a thread that loaded each pixel's key
// before its store spent the draw waiting on those loads one at a time (four times the post-processing's device time
// for 64 frames of 480x640); the scan streams 4 bytes per pixel at full bandwidth.
//
// The rasteriser is __host__ __device__: ekp_debug_raster_host / ekp_debug_draw_host run the same code on the CPU, so
// tests pin it to cv2 without a GPU.  They are test hooks, not a CPU path of ekp_draw_humans.
#include <math.h>
#include <string.h>

#include "common.cuh"

namespace ekp {

#define HD __host__ __device__ __forceinline__

static const int kPrimsPerHuman = EKP_NUM_PART + 17;  // 18 part markers, then the 17 limbs of CocoPairsRender
static_assert(EKP_LIMIT_HUMANS * kPrimsPerHuman < 65536, "s + 1 must fit the low 16 bits of a key");

// lib/utils/common.py CocoColors, written to channels 0, 1, 2 in tuple order as cv2 does
__constant__ const unsigned char kColorsDev[18][3] = {
    {255, 0, 0},   {255, 85, 0},  {255, 170, 0}, {255, 255, 0}, {170, 255, 0}, {85, 255, 0},  {0, 255, 0},   {0, 255, 85},
    {0, 255, 170}, {0, 255, 255}, {0, 170, 255}, {0, 85, 255},  {0, 0, 255},   {85, 0, 255},  {170, 0, 255}, {255, 0, 255},
    {255, 0, 170}, {255, 0, 85}};
static const unsigned char kColorsHost[18][3] = {
    {255, 0, 0},   {255, 85, 0},  {255, 170, 0}, {255, 255, 0}, {170, 255, 0}, {85, 255, 0},  {0, 255, 0},   {0, 255, 85},
    {0, 255, 170}, {0, 255, 255}, {0, 170, 255}, {0, 85, 255},  {0, 0, 255},   {85, 0, 255},  {170, 0, 255}, {255, 0, 255},
    {255, 0, 170}, {255, 0, 85}};
// CocoPairsRender = CocoPairs[:-2] (the first 17 limbs of pafprocess.h:16-24)
__constant__ const signed char kRenderDev[17][2] = {{1, 2}, {1, 5}, {2, 3},  {3, 4},  {5, 6},   {6, 7},  {1, 8},   {8, 9}, {9, 10},
                                                    {1, 11}, {11, 12}, {12, 13}, {1, 0}, {0, 14}, {14, 16}, {0, 15}, {15, 17}};
[[maybe_unused]] static const signed char kRenderHost[17][2] = {{1, 2}, {1, 5}, {2, 3},  {3, 4},  {5, 6},   {6, 7},  {1, 8},   {8, 9}, {9, 10},
                                               {1, 11}, {11, 12}, {12, 13}, {1, 0}, {0, 14}, {14, 16}, {0, 15}, {15, 17}};
// cv2.circle(img, c, 3, colour, thickness=3, lineType=8): 96 pixels in |dx|, |dy| <= 5, bit dx + 5 of row dy + 5.  The
// centre pixel is not painted.  Clipped to the frame this equals cv2 for every centre at most one pixel outside it, which
// covers every centre draw_humans forms (tests/test_draw_humans.py pins it to cv2).
__constant__ const unsigned short kRingDev[11] = {0xf8, 0x1fc, 0x3fe, 0x7ff, 0x7ff, 0x7df, 0x7ff, 0x7ff, 0x3fe, 0x1fc, 0xf8};
[[maybe_unused]] static const unsigned short kRingHost[11] = {0xf8, 0x1fc, 0x3fe, 0x7ff, 0x7ff, 0x7df, 0x7ff, 0x7ff, 0x3fe, 0x1fc, 0xf8};

#ifdef __CUDA_ARCH__
#define TABLE(name) name##Dev
#else
#define TABLE(name) name##Host
#endif

// cv2 drawing.cpp fixed point: XY_SHIFT = 16
static const int kShift = 16;
static const long long kOne = 1ll << kShift;

template <class T>
HD void swap2(T& a, T& b) { T t = a; a = b; b = t; }
HD long long min2(long long a, long long b) { return a < b ? a : b; }
HD long long max2(long long a, long long b) { return a > b ? a : b; }

// Put: put(x, y) for one pixel inside the frame, span(y, x1, x2) for x1..x2 inside the frame (empty when x1 > x2)
#pragma nv_exec_check_disable  // Put is a __device__ functor in the kernels, a host one in the test hooks
template <class Put>
HD void put_clipped(Put& put, int x, int y, int H, int W) {
    if (0 <= x && x < W && 0 <= y && y < H) put.put(x, y);
}

// clipLine(Size2l, Point2l&, Point2l&) in 16.16 fixed point; false when the segment misses the frame
HD bool clip_line(long long w, long long h, long long& x1, long long& y1, long long& x2, long long& y2) {
    const long long right = w - 1, bottom = h - 1;
    int c1 = (x1 < 0) + (x1 > right) * 2 + (y1 < 0) * 4 + (y1 > bottom) * 8;
    int c2 = (x2 < 0) + (x2 > right) * 2 + (y2 < 0) * 4 + (y2 > bottom) * 8;
    if ((c1 & c2) == 0 && (c1 | c2) != 0) {
        long long a;
        if (c1 & 12) {
            a = c1 < 8 ? 0 : bottom;
            x1 += (long long) ((double) (a - y1) * (double) (x2 - x1) / (double) (y2 - y1));
            y1 = a;
            c1 = (x1 < 0) + (x1 > right) * 2;
        }
        if (c2 & 12) {
            a = c2 < 8 ? 0 : bottom;
            x2 += (long long) ((double) (a - y2) * (double) (x2 - x1) / (double) (y2 - y1));
            y2 = a;
            c2 = (x2 < 0) + (x2 > right) * 2;
        }
        if ((c1 & c2) == 0 && (c1 | c2) != 0) {
            if (c1) {
                a = c1 == 1 ? 0 : right;
                y1 += (long long) ((double) (a - x1) * (double) (y2 - y1) / (double) (x2 - x1));
                x1 = a;
                c1 = 0;
            }
            if (c2) {
                a = c2 == 1 ? 0 : right;
                y2 += (long long) ((double) (a - x2) * (double) (y2 - y1) / (double) (x2 - x1));
                x2 = a;
                c2 = 0;
            }
        }
    }
    return (c1 | c2) == 0;
}

// Line2: the 8-connected outline segment between two 16.16 points, clipped first
template <class Put>
HD void line2(long long x1, long long y1, long long x2, long long y2, int H, int W, Put& put) {
    if (!clip_line((long long) W << kShift, (long long) H << kShift, x1, y1, x2, y2)) return;
    long long dx = x2 - x1, dy = y2 - y1;
    const long long ax = dx < 0 ? -dx : dx, ay = dy < 0 ? -dy : dy;
    long long x_step, y_step;
    int ecount;
    if (ax > ay) {
        if (dx < 0) { dy = -dy; swap2(x1, x2); swap2(y1, y2); }
        x_step = kOne;
        y_step = dy * kOne / (ax | 1);
        ecount = (int) ((x2 - x1) >> kShift);
    } else {
        if (dy < 0) { dx = -dx; swap2(x1, x2); swap2(y1, y2); }
        x_step = dx * kOne / (ay | 1);
        y_step = kOne;
        ecount = (int) ((y2 - y1) >> kShift);
    }
    x1 += kOne >> 1;
    y1 += kOne >> 1;
    put_clipped(put, (int) ((x2 + (kOne >> 1)) >> kShift), (int) ((y2 + (kOne >> 1)) >> kShift), H, W);
    if (ax > ay) {
        x1 >>= kShift;
        for (; ecount >= 0; ecount--, x1++, y1 += y_step) put_clipped(put, (int) x1, (int) (y1 >> kShift), H, W);
    } else {
        y1 >>= kShift;
        for (; ecount >= 0; ecount--, x1 += x_step, y1++) put_clipped(put, (int) (x1 >> kShift), (int) y1, H, W);
    }
}

// FillConvexPoly(img, v, 4, colour, LINE_8, XY_SHIFT): the outline through Line2, then the scanline spans
#pragma nv_exec_check_disable  // Put is a __device__ functor in the kernels, a host one in the test hooks
template <class Put>
HD void fill_quad(const long long (*v)[2], int H, int W, Put& put) {
    const int npts = 4;
    const long long delta = kOne >> 1;
    long long xmin = v[0][0], xmax = v[0][0], ymin = v[0][1], ymax = v[0][1];
    int imin = 0;
    long long p0x = v[npts - 1][0], p0y = v[npts - 1][1];
    for (int i = 0; i < npts; i++) {
        if (v[i][1] < ymin) { ymin = v[i][1]; imin = i; }
        ymax = max2(ymax, v[i][1]);
        xmax = max2(xmax, v[i][0]);
        xmin = min2(xmin, v[i][0]);
        line2(p0x, p0y, v[i][0], v[i][1], H, W, put);
        p0x = v[i][0]; p0y = v[i][1];
    }
    xmin = (xmin + delta) >> kShift;
    xmax = (xmax + delta) >> kShift;
    ymin = (ymin + delta) >> kShift;
    ymax = (ymax + delta) >> kShift;
    if ((int) xmax < 0 || (int) ymax < 0 || (int) xmin >= W || (int) ymin >= H) return;
    ymax = min2(ymax, H - 1);
    struct { int idx, di; long long x, dx; int ye; } edge[2];
    edge[0].idx = edge[1].idx = imin;
    int y = (int) ymin;
    edge[0].ye = edge[1].ye = y;
    edge[0].di = 1;
    edge[1].di = npts - 1;
    edge[0].x = edge[1].x = -kOne;
    edge[0].dx = edge[1].dx = 0;
    int edges = npts;
    do {
        for (int i = 0; i < 2; i++) {
            if (y >= edge[i].ye) {
                int idx0 = edge[i].idx, di = edge[i].di;
                int idx = idx0 + di;
                if (idx >= npts) idx -= npts;
                for (; edges-- > 0;) {
                    const int ty = (int) ((v[idx][1] + delta) >> kShift);
                    if (ty > y) {
                        const long long xs = v[idx0][0], xe = v[idx][0];
                        edge[i].ye = ty;
                        edge[i].dx = ((xe - xs) * 2 + ((long long) ty - y)) / (2 * ((long long) ty - y));
                        edge[i].x = xs;
                        edge[i].idx = idx;
                        break;
                    }
                    idx0 = idx;
                    idx += di;
                    if (idx >= npts) idx -= npts;
                }
            }
        }
        if (edges < 0) break;
        if (y >= 0) {
            const int left = edge[0].x > edge[1].x ? 1 : 0, right = 1 - left;
            int xx1 = (int) ((edge[left].x + delta) >> kShift);
            int xx2 = (int) ((edge[right].x + delta) >> kShift);
            if (xx2 >= 0 && xx1 < W) {
                if (xx1 < 0) xx1 = 0;
                if (xx2 >= W) xx2 = W - 1;
                put.span(y, xx1, xx2);
            }
        }
        edge[0].x += edge[0].dx;
        edge[1].x += edge[1].dx;
    } while (++y <= (int) ymax);
}

// Circle(img, center, radius, colour, fill = 1): the round cap of a thick LINE_8 line
#pragma nv_exec_check_disable  // Put is a __device__ functor in the kernels, a host one in the test hooks
template <class Put>
HD void filled_circle(int cx, int cy, int radius, int H, int W, Put& put) {
    int err = 0, dx = radius, dy = 0, plus = 1, minus = (radius << 1) - 1;
    while (dx >= dy) {
        const int y11 = cy - dy, y12 = cy + dy, y21 = cy - dx, y22 = cy + dx;
        int x11 = cx - dx, x12 = cx + dx, x21 = cx - dy, x22 = cx + dy;
        if (x11 < W && x12 >= 0 && y21 < H && y22 >= 0) {
            x11 = x11 > 0 ? x11 : 0;
            x12 = x12 < W - 1 ? x12 : W - 1;
            if ((unsigned) y11 < (unsigned) H) put.span(y11, x11, x12);
            if ((unsigned) y12 < (unsigned) H) put.span(y12, x11, x12);
            if (x21 < W && x22 >= 0) {
                x21 = x21 > 0 ? x21 : 0;
                x22 = x22 < W - 1 ? x22 : W - 1;
                if ((unsigned) y21 < (unsigned) H) put.span(y21, x21, x22);
                if ((unsigned) y22 < (unsigned) H) put.span(y22, x21, x22);
            }
        }
        dy++;
        err += plus;
        plus += 2;
        const int mask = (err <= 0) - 1;
        err -= minus & mask;
        dx += mask;
        minus -= mask & 2;
    }
}

// cv2.line(img, p0, p1, colour, 3) = ThickLine(thickness 3, LINE_8, both caps, shift 0)
template <class Put>
HD void thick_line3(int x0, int y0, int x1, int y1, int H, int W, Put& put) {
    const long long p0x = (long long) x0 << kShift, p0y = (long long) y0 << kShift;
    const long long p1x = (long long) x1 << kShift, p1y = (long long) y1 << kShift;
    const double inv_one = 1. / (double) kOne;
    const double dx = (double) (p0x - p1x) * inv_one, dy = (double) (p1y - p0y) * inv_one;
    double r = dx * dx + dy * dy;
    const int thickness = 3 << (kShift - 1), odd = 1;
    if (fabs(r) > 2.220446049250313e-16 /* DBL_EPSILON */) {
        r = ((double) thickness + odd * (double) kOne * 0.5) / sqrt(r);
        const long long dpx = (long long) rint(dy * r), dpy = (long long) rint(dx * r);  // cvRound: nearest, ties to even
        const long long v[4][2] = {{p0x + dpx, p0y + dpy}, {p0x - dpx, p0y - dpy}, {p1x - dpx, p1y - dpy}, {p1x + dpx, p1y + dpy}};
        fill_quad(v, H, W, put);
    }
    const int radius = (thickness + (int) (kOne >> 1)) >> kShift;
    filled_circle(x0, y0, radius, H, W, put);
    filled_circle(x1, y1, radius, H, W, put);
}

template <class Put>
HD void ring3(int cx, int cy, int H, int W, Put& put) {
    for (int dy = -5; dy <= 5; dy++) {
        const int y = cy + dy;
        if (y < 0 || y >= H) continue;
        const unsigned row = TABLE(kRing)[dy + 5];
        for (int dx = -5; dx <= 5; dx++)
            if ((row >> (dx + 5)) & 1u) put_clipped(put, cx + dx, y, H, W);
    }
}

// draw_humans' centre (int(body_part.x * image_w + 0.5), ...) with body_part.x = float(px) / map_w as the reference
// forms it in Python doubles: a division, a multiplication and an addition, each rounded.  The Makefile builds with
// -fmad=false (device) and -ffp-contract=off (host), so the multiply-add is not contracted into an FMA.
HD int centre(int p, int map_n, int n) { return (int) ((double) p / (double) map_n * (double) n + 0.5); }

struct Prim {
    int kind;  // 0: nothing, 1: part marker at (x0, y0), 2: limb (x0, y0) - (x1, y1)
    int x0, y0, x1, y1, color;
};

// primitive j (0..34) of one human's parts [18]
HD Prim prim_of(const ekp_peak* parts, int j, int map_h, int map_w, int H, int W) {
    Prim p = {0, 0, 0, 0, 0, 0};
    if (j < EKP_NUM_PART) {
        if (parts[j].id < 0) return p;
        p.kind = 1;
        p.x0 = centre(parts[j].x, map_w, W);
        p.y0 = centre(parts[j].y, map_h, H);
        p.color = j;
    } else {
        const int l = j - EKP_NUM_PART, a = TABLE(kRender)[l][0], b = TABLE(kRender)[l][1];
        if (parts[a].id < 0 || parts[b].id < 0) return p;
        p.kind = 2;
        p.x0 = centre(parts[a].x, map_w, W);
        p.y0 = centre(parts[a].y, map_h, H);
        p.x1 = centre(parts[b].x, map_w, W);
        p.y1 = centre(parts[b].y, map_h, H);
        p.color = l;
    }
    return p;
}

template <class Put>
HD void raster(const Prim& p, int H, int W, Put& put) {
    if (p.kind == 1) ring3(p.x0, p.y0, H, W, put);
    else if (p.kind == 2) thick_line3(p.x0, p.y0, p.x1, p.y1, H, W, put);
}

// ---- device: cover, then paint ------------------------------------------------------------------------------------
struct DrawParams {  // of pass 1
    const unsigned char* records;  // [n] packed result records of the last run (ResultLayout)
    ResultLayout lay;
    int max_humans, map_h, map_w;
    int H, W;
    unsigned* keys;                // [n][H][W]
    unsigned epoch;                // 1 .. 65535
};

struct Cover {
    unsigned* key;
    int W;
    unsigned tag;
    __device__ void put(int x, int y) { atomicMax(key + (size_t) y * W + x, tag); }
    __device__ void span(int y, int x1, int x2) { for (int x = x1; x <= x2; x++) put(x, y); }
};
// pass 1: one thread per primitive s of image blockIdx.y
__global__ void __launch_bounds__(128) draw_cover_kernel(const DrawParams P) {
    const int img = blockIdx.y;
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned char* rec = P.records + P.lay.stride * (size_t) img;
    const int num = min(*reinterpret_cast<const int*>(rec), P.max_humans);
    if (s >= num * kPrimsPerHuman) return;
    const int k = s / kPrimsPerHuman, j = s - k * kPrimsPerHuman;
    const ekp_peak* parts = reinterpret_cast<const ekp_peak*>(rec + P.lay.off_hparts) + (size_t) k * EKP_NUM_PART;
    const Prim p = prim_of(parts, j, P.map_h, P.map_w, P.H, P.W);
    if (!p.kind) return;
    Cover put{P.keys + (size_t) img * P.H * P.W, P.W, P.epoch << 16 | (unsigned) (s + 1)};
    raster(p, P.H, P.W, put);
}

__device__ __forceinline__ void paint1(unsigned key, unsigned epoch, unsigned char* px) {
    if (key >> 16 != epoch) return;  // no primitive of this draw covers the pixel
    const int j = (int) ((key & 0xffffu) - 1) % kPrimsPerHuman;
    const unsigned char* c = kColorsDev[j < EKP_NUM_PART ? j : j - EKP_NUM_PART];
    px[0] = c[0]; px[1] = c[1]; px[2] = c[2];
}

// pass 2: keys [pixels] (16-byte aligned) -> colours of the frames [pixels][3] where this draw covered the pixel
__global__ void __launch_bounds__(256) draw_paint_kernel(const unsigned* __restrict__ keys, unsigned char* __restrict__ frames,
                                                         size_t pixels, unsigned epoch) {
    const size_t quads = pixels / 4, stride = (size_t) gridDim.x * blockDim.x;
    for (size_t q = (size_t) blockIdx.x * blockDim.x + threadIdx.x; q < quads; q += stride) {
        const uint4 k = __ldcs(reinterpret_cast<const uint4*>(keys) + q);   // read once: do not keep it in L2
        unsigned char* px = frames + 12 * q;
        paint1(k.x, epoch, px); paint1(k.y, epoch, px + 3); paint1(k.z, epoch, px + 6); paint1(k.w, epoch, px + 9);
    }
    if (blockIdx.x == 0 && threadIdx.x < (pixels & 3)) {
        const size_t o = 4 * quads + threadIdx.x;
        paint1(keys[o], epoch, frames + 3 * o);
    }
}

cudaError_t launch_draw(const unsigned char* records, const ResultLayout& lay, int max_humans, int map_h, int map_w,
                        unsigned char* frames, int n, int H, int W, unsigned* keys, unsigned epoch, cudaStream_t stream) {
    DrawParams P;
    P.records = records; P.lay = lay; P.max_humans = max_humans; P.map_h = map_h; P.map_w = map_w;
    P.H = H; P.W = W; P.keys = keys; P.epoch = epoch;
    const dim3 grid((unsigned) ((max_humans * kPrimsPerHuman + 127) / 128), (unsigned) n);
    draw_cover_kernel<<<grid, 128, 0, stream>>>(P);
    int dev = 0, sms = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess) return e;
    const size_t pixels = (size_t) n * H * W, want = (pixels / 4 + 255) / 256;
    const int blocks = (int) (want < 1 ? 1 : (want < (size_t) sms * 8 ? want : (size_t) sms * 8));  // 8 x 256 threads fill an SM
    draw_paint_kernel<<<blocks, 256, 0, stream>>>(keys, frames, pixels, epoch);
    return cudaGetLastError();
}

// ---- host: the same rasteriser, serially in drawing order (test hooks) ------------------------------------------------
struct HostMask {
    unsigned char* m;
    int W;
    void put(int x, int y) { m[(size_t) y * W + x] = 1; }
    void span(int y, int x1, int x2) { for (int x = x1; x <= x2; x++) put(x, y); }
};
struct HostPaint {
    unsigned char* px;
    int W;
    const unsigned char* c;
    void put(int x, int y) { memcpy(px + 3 * ((size_t) y * W + x), c, 3); }
    void span(int y, int x1, int x2) { for (int x = x1; x <= x2; x++) put(x, y); }
};

void debug_raster_host(int kind, int x0, int y0, int x1, int y1, int H, int W, unsigned char* mask) {
    const Prim p = {kind, x0, y0, x1, y1, 0};
    HostMask put{mask, W};
    raster(p, H, W, put);
}

void debug_draw_host(const int* num_humans, const ekp_peak* parts, int max_humans, int map_h, int map_w,
                     unsigned char* frames, int n, int H, int W) {
    for (int i = 0; i < n; i++) {
        const int num = num_humans[i] < max_humans ? num_humans[i] : max_humans;
        unsigned char* px = frames + (size_t) i * H * W * 3;
        for (int k = 0; k < num; k++) {
            const ekp_peak* hp = parts + ((size_t) i * max_humans + k) * EKP_NUM_PART;
            for (int j = 0; j < kPrimsPerHuman; j++) {
                const Prim p = prim_of(hp, j, map_h, map_w, H, W);
                HostPaint put{px, W, kColorsHost[p.color]};
                raster(p, H, W, put);
            }
        }
    }
}

}  // namespace ekp
