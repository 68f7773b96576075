// coco_eval.cu -- pycocotools' COCOeval for iouType 'keypoints', one category, on the device (ekp_coco_eval_kpts):
// the precision [T, R, A], recall [T, A] and scores [T, R, A] arrays of accumulate(), bit for bit.
//
// Specification: include/ekpose_b200.h ("COCO keypoint evaluation") and DESIGN.md section 8.  The work is four steps:
//   1. coco_match_kernel, one block per image: the stable order of its detections by score (truncated to max_det), the
//      float64 OKS matrix of those detections against the image's ground truth (pycocotools' computeOks, numpy's
//      summation order included), the detections' areas (loadRes), and one greedy walk (evaluateImg) per area range and
//      threshold, one thread per walk.  Per kept detection it writes a tp and an fp bit over the A x T <= 32 curves, its
//      score and its global sort key into slot img * max_det + rank; slots past the image's kept count get the largest
//      key and no bits.
//   2. An LSD radix sort of all slots by key, 8 bits per pass (histogram, one-block scan, stable scatter through
//      cub::BlockRadixSort), so equal scores keep slot order, i.e. image order then rank: accumulate()'s mergesort of
//      the concatenated detections.
//   3. Per chunk of kCocoChunk sorted positions: the masks in sorted order and their per-curve counts; one block scans
//      the chunk counts (and sums nd and npig); per chunk the precision maximum of each curve.
//   4. One block per curve: the suffix maxima of the chunk maxima (the precision envelope), and per recall threshold the
//      searchsorted position as the position of the k-th true positive, k the least count with k / npig >= recThr.
// Steps 1, 3 and 4 are __host__ __device__: ekp_debug_coco_eval_host runs the same code serially on the CPU (a test hook,
// not a CPU path of the evaluation), with std::stable_sort on the same keys in place of the radix sort.
#include <math.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include <cub/block/block_radix_sort.cuh>
#include <cub/block/block_scan.cuh>

#include "common.cuh"

namespace ekp {

#define HD __host__ __device__ __forceinline__

static const int kKp = 17;
static const int kMatchThreads = 128;
static const int kSortThreads = 256, kSortItems = 8, kSortTile = kSortThreads * kSortItems;  // 2048 keys per tile
static const int kSortPasses = 8;                                                           // 64-bit keys, 8 bits a pass
static const int kScanThreads = 1024;
static const int kCocoChunk = 512;   // sorted positions per accumulate chunk
static const int kChunkThreads = 256;
static const int kCurveThreads = 128;
static const size_t kCocoSmemMax = 227 * 1024;
static const unsigned long long kPadKey = ~0ull;   // slots past an image's kept detections: sorted after every score

HD void cbar() {
#ifdef __CUDA_ARCH__
    __syncthreads();
#endif
}
HD void or_bits(unsigned* word, unsigned bits) {
#ifdef __CUDA_ARCH__
    atomicOr(word, bits);
#else
    *word |= bits;
#endif
}
HD unsigned long long dbits(double v) {
#ifdef __CUDA_ARCH__
    return (unsigned long long) __double_as_longlong(v);
#else
    unsigned long long u;
    memcpy(&u, &v, 8);
    return u;
#endif
}

// Ascending key = descending score, total over all bit patterns: -0.0 is first made +0.0 (numpy's comparisons see them
// equal), then the usual order-preserving map of the IEEE bits, inverted.
HD unsigned long long score_key(double s) {
    const unsigned long long u = dbits(s + 0.0);
    const unsigned long long ord = (u >> 63) ? ~u : (u | 0x8000000000000000ull);
    return ~ord;
}

// numpy's float64 add.reduce of a contiguous array of n <= 17 terms (pairwise_sum: sequential below 8 terms, else eight
// accumulators over the multiple-of-8 prefix, a fixed tree, then the rest in order)
HD double np_sum(const double* a, int n) {
    if (n < 8) {
        double r = -0.0;
        for (int i = 0; i < n; i++) r += a[i];
        return r;
    }
    double r[8];
    for (int j = 0; j < 8; j++) r[j] = a[j];
    int i = 8;
    for (; i < n - (n % 8); i += 8)
        for (int j = 0; j < 8; j++) r[j] += a[i + j];
    double res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
    for (; i < n; i++) res += a[i];
    return res;
}

// computeOks for one (detection, ground truth) pair: g / d point at 17 (x, y, v) triples, bb at the gt's bbox
HD double coco_oks(const double* d, const double* g, const double* bb, double garea, const double* var) {
    int k1 = 0;
    for (int j = 0; j < kKp; j++) k1 += g[3 * j + 2] > 0;
    const double x0 = bb[0] - bb[2], x1 = bb[0] + bb[2] * 2, y0 = bb[1] - bb[3], y1 = bb[1] + bb[3] * 2;
    const double den = garea + 2.220446049250313e-16;   // gt['area'] + np.spacing(1)
    double t[kKp];
    int n = 0;
    for (int j = 0; j < kKp; j++) {
        double dx, dy;
        if (k1 > 0) {
            if (!(g[3 * j + 2] > 0)) continue;
            dx = d[3 * j] - g[3 * j];
            dy = d[3 * j + 1] - g[3 * j + 1];
        } else {
            const double ax = x0 - d[3 * j], bx = d[3 * j] - x1, ay = y0 - d[3 * j + 1], by = d[3 * j + 1] - y1;
            dx = (ax > 0 ? ax : 0.0) + (bx > 0 ? bx : 0.0);
            dy = (ay > 0 ? ay : 0.0) + (by > 0 ? by : 0.0);
        }
        const double e = (dx * dx + dy * dy) / var[j] / den / 2;
        t[n++] = exp(-e);
    }
    return np_sum(t, n) / n;
}

// loadRes' area of a detection: over all 17 keypoints, absent (0, 0, 0) triples included
HD double coco_dt_area(const double* d) {
    double x0 = d[0], x1 = d[0], y0 = d[1], y1 = d[1];
    for (int j = 1; j < kKp; j++) {
        const double x = d[3 * j], y = d[3 * j + 1];
        x0 = x < x0 ? x : x0; x1 = x > x1 ? x : x1;
        y0 = y < y0 ? y : y0; y1 = y > y1 ? y : y1;
    }
    return (x1 - x0) * (y1 - y0);
}

struct CocoArgs {
    ekp_coco_gt gt;
    ekp_coco_dt dt;
    int max_gt, max_dt, n_img, max_det, T, R, A;
    const double* iou;     // [T]
    const double* rec;     // [R]
    const double* area;    // [A][2]
    double var[kKp];       // oks_vars
    ekp_coco_eval_out out;
    // workspace
    unsigned* tpm;         // [S] per slot: bit a * T + t = true positive of curve (a, t)
    unsigned* fpm;         // [S]
    double* sscore;        // [S] the slot's score as given
    unsigned long long* key[2];  // [S] sort keys, ping-pong
    int* val[2];                 // [S] slot indices riding along
    int* kept;             // [n_img] kept detections
    int* npig_img;         // [n_img][A] non-ignored ground truths
    unsigned* hist;        // [256][n_tiles] sort histograms, then their exclusive scan
    unsigned* stp;         // [S] tp masks in sorted order
    unsigned* sfp;         // [S]
    int* ccnt;             // [n_chunks][32][2] per chunk and curve: tp, fp counts
    int* cpre;             // [n_chunks][32][2] their exclusive prefix over chunks
    double* cmax;          // [n_chunks][32] per chunk: the largest precision of its positions < nd
    double* csuf;          // [32][n_chunks + 1] suffix maxima of cmax
    int* tot;              // [0] nd, [1 .. A] npig, [1 + A + 2c + k] total tp / fp of curve c
    int S, n_tiles, n_chunks;
};

// ---- workspace ------------------------------------------------------------------------------------------------------
struct CocoSizes { long long S, n_tiles, n_chunks; };
static CocoSizes coco_sizes(long long n_img, long long max_det) {
    CocoSizes z;
    z.S = n_img * max_det;
    z.n_tiles = (z.S + kSortTile - 1) / kSortTile;
    z.n_chunks = (z.S + kCocoChunk - 1) / kCocoChunk;
    return z;
}
// Carves the workspace out of `base` (nullptr: only sizes it); returns its bytes.
static size_t coco_ws_layout(long long n_img, long long max_det, int A, unsigned char* base, CocoArgs* a) {
    const CocoSizes z = coco_sizes(n_img, max_det);
    size_t off = 0;
    auto take = [&](size_t bytes) { unsigned char* p = base ? base + off : nullptr; off += (bytes + 255) & ~(size_t) 255; return p; };
    CocoArgs t = {};
    t.tpm = (unsigned*) take(4 * z.S);
    t.fpm = (unsigned*) take(4 * z.S);
    t.sscore = (double*) take(8 * z.S);
    t.key[0] = (unsigned long long*) take(8 * z.S);
    t.key[1] = (unsigned long long*) take(8 * z.S);
    t.val[0] = (int*) take(4 * z.S);
    t.val[1] = (int*) take(4 * z.S);
    t.kept = (int*) take(4 * n_img);
    t.npig_img = (int*) take(4 * n_img * A);
    t.hist = (unsigned*) take(4 * 256 * z.n_tiles);
    t.stp = (unsigned*) take(4 * z.S);
    t.sfp = (unsigned*) take(4 * z.S);
    t.ccnt = (int*) take(4 * 64 * z.n_chunks);
    t.cpre = (int*) take(4 * 64 * z.n_chunks);
    t.cmax = (double*) take(8 * 32 * z.n_chunks);
    t.csuf = (double*) take(8 * 32 * (z.n_chunks + 1));
    t.tot = (int*) take(4 * (1 + 32 + 64));
    if (a) {
        a->tpm = t.tpm; a->fpm = t.fpm; a->sscore = t.sscore;
        a->key[0] = t.key[0]; a->key[1] = t.key[1]; a->val[0] = t.val[0]; a->val[1] = t.val[1];
        a->kept = t.kept; a->npig_img = t.npig_img; a->hist = t.hist; a->stp = t.stp; a->sfp = t.sfp;
        a->ccnt = t.ccnt; a->cpre = t.cpre; a->cmax = t.cmax; a->csuf = t.csuf; a->tot = t.tot;
        a->S = (int) z.S; a->n_tiles = (int) z.n_tiles; a->n_chunks = (int) z.n_chunks;
    }
    return off;
}
size_t coco_eval_ws_bytes(long long n_img, long long max_det, int A) { return coco_ws_layout(n_img, max_det, A, nullptr, nullptr); }

// ---- step 1: one image ----------------------------------------------------------------------------------------------
struct CocoImgWork {     // shared memory on the device
    double* oks;         // [max_det][max_gt]
    double* dtarea;      // [max_det]
    unsigned long long* dkey;  // [max_dt]
    int* sel;            // [max_det] row of the detection of each rank
    unsigned char* gtm;  // [32][max_gt] per walk: ground truth matched
    unsigned* bits;      // [2][max_det] tp / fp masks
};
HD size_t coco_img_layout(int max_gt, int max_dt, int max_det, unsigned char* base, CocoImgWork* w) {
    size_t off = 0;
    auto take = [&](size_t bytes) { unsigned char* p = base ? base + off : nullptr; off += (bytes + 15) & ~(size_t) 15; return p; };
    CocoImgWork t;
    t.oks = (double*) take(sizeof(double) * max_det * max_gt);
    t.dtarea = (double*) take(sizeof(double) * max_det);
    t.dkey = (unsigned long long*) take(sizeof(unsigned long long) * max_dt);
    t.sel = (int*) take(sizeof(int) * max_det);
    t.bits = (unsigned*) take(sizeof(unsigned) * 2 * max_det);
    t.gtm = (unsigned char*) take((size_t) 32 * max_gt);
    if (w) *w = t;
    return off;
}

HD bool outside(double area, const double* rng) { return area < rng[0] || area > rng[1]; }

HD void coco_image(const CocoArgs& P, int img, const CocoImgWork& W, int tid, int nt) {
    const int MG = P.max_gt, MD = P.max_dt, K = P.max_det;
    const int nd = min(max(P.dt.count[img], 0), MD), ng = min(max(P.gt.count[img], 0), MG);
    const int kept = min(nd, K);
    const double* dkp = P.dt.keypoints + (size_t) img * MD * 3 * kKp;
    const double* dsc = P.dt.score + (size_t) img * MD;
    const double* gkp = P.gt.keypoints + (size_t) img * MG * 3 * kKp;
    const double* gbb = P.gt.bbox + (size_t) img * MG * 4;
    const double* gar = P.gt.area + (size_t) img * MG;
    const int* gcr = P.gt.iscrowd + (size_t) img * MG;
    const int* gig = P.gt.ignore + (size_t) img * MG;
    // the stable order by score: rank = detections before this one in (key, row) order
    for (int j = tid; j < nd; j += nt) W.dkey[j] = score_key(dsc[j]);
    for (int d = tid; d < K; d += nt) { W.bits[d] = 0; W.bits[K + d] = 0; }
    cbar();
    for (int j = tid; j < nd; j += nt) {
        const unsigned long long kj = W.dkey[j];
        int r = 0;
        for (int q = 0; q < nd; q++) r += W.dkey[q] < kj || (W.dkey[q] == kj && q < j);
        if (r < K) W.sel[r] = j;
    }
    cbar();
    for (int u = tid; u < kept * ng; u += nt) {
        const int d = u / ng, g = u - d * ng;
        W.oks[d * MG + g] = coco_oks(dkp + (size_t) W.sel[d] * 3 * kKp, gkp + (size_t) g * 3 * kKp, gbb + 4 * g, gar[g], P.var);
    }
    for (int d = tid; d < kept; d += nt) W.dtarea[d] = coco_dt_area(dkp + (size_t) W.sel[d] * 3 * kKp);
    for (int a = tid; a < P.A; a += nt) {
        int c = 0;
        for (int g = 0; g < ng; g++) c += !(gig[g] || outside(gar[g], P.area + 2 * a));
        P.npig_img[(size_t) img * P.A + a] = c;
    }
    cbar();
    // evaluateImg: walk c = a * T + t over the detections in rank order; the ground truths in the order of the stable
    // sort by _ignore (the non-ignored ones first, each group in row order)
    for (int c = tid; c < P.A * P.T; c += nt) {
        const int a = c / P.T, t = c - a * P.T;
        const double* rng = P.area + 2 * a;
        const double thr = P.iou[t];
        unsigned char* gtm = W.gtm + (size_t) c * MG;
        for (int g = 0; g < ng; g++) gtm[g] = 0;
        for (int d = 0; d < kept; d++) {
            double iou = 1.0 - 1e-10 < thr ? 1.0 - 1e-10 : thr;   // min([t, 1 - 1e-10])
            int m = -1, mig = 0;
            bool stop = false;
            for (int pass = 0; pass < 2 && !stop; pass++) {
                for (int g = 0; g < ng; g++) {
                    const int ig = gig[g] || outside(gar[g], rng);
                    if (ig != pass) continue;
                    if (gtm[g] && !gcr[g]) continue;
                    if (m > -1 && mig == 0 && ig == 1) { stop = true; break; }
                    const double o = W.oks[d * MG + g];
                    if (o < iou) continue;
                    iou = o; m = g; mig = ig;
                }
            }
            int dig;
            if (m >= 0) { dig = mig; gtm[m] = 1; }
            else dig = outside(W.dtarea[d], rng);
            if (!dig) or_bits(&W.bits[(m >= 0 ? 0 : K) + d], 1u << c);
            const size_t o = (((size_t) img * P.A + a) * P.T + t) * K + d;
            if (P.out.dt_match) P.out.dt_match[o] = m;
            if (P.out.dt_ignore) P.out.dt_ignore[o] = dig;
        }
        for (int d = kept; d < K; d++) {
            const size_t o = (((size_t) img * P.A + a) * P.T + t) * K + d;
            if (P.out.dt_match) P.out.dt_match[o] = -1;
            if (P.out.dt_ignore) P.out.dt_ignore[o] = 0;
        }
    }
    if (P.out.oks)
        for (int u = tid; u < K * MG; u += nt) {
            const int d = u / MG, g = u - d * MG;
            P.out.oks[(size_t) img * K * MG + u] = d < kept && g < ng ? W.oks[d * MG + g] : 0.0;
        }
    cbar();
    for (int d = tid; d < K; d += nt) {
        const size_t s = (size_t) img * K + d;
        P.tpm[s] = W.bits[d];
        P.fpm[s] = W.bits[K + d];
        P.sscore[s] = d < kept ? dsc[W.sel[d]] : 0.0;
        P.key[0][s] = d < kept ? W.dkey[W.sel[d]] : kPadKey;
        P.val[0][s] = (int) s;
    }
    if (tid == 0) P.kept[img] = kept;
}

// ---- step 3: chunks of sorted positions -----------------------------------------------------------------------------
// the masks of chunk ch in sorted order (order = the sorted slot indices) and their per-curve counts
HD void coco_chunk_counts(const CocoArgs& P, const int* order, int ch, unsigned* stage, int tid, int nt) {
    const int base = ch * kCocoChunk, len = min(kCocoChunk, P.S - base);
    for (int j = tid; j < len; j += nt) {
        const int s = order[base + j];
        const unsigned tp = P.tpm[s], fp = P.fpm[s];
        P.stp[base + j] = tp; P.sfp[base + j] = fp;
        stage[j] = tp; stage[kCocoChunk + j] = fp;
    }
    cbar();
    for (int u = tid; u < 64; u += nt) {
        const int c = u >> 1;
        const unsigned* m = stage + (u & 1) * kCocoChunk;
        int n = 0;
        for (int j = 0; j < len; j++) n += (m[j] >> c) & 1u;
        P.ccnt[(size_t) ch * 64 + u] = n;
    }
}

// precision at a position with tp / fp counts so far: tp / ((fp + tp) + np.spacing(1))
HD double prec(int tp, int fp) { return (double) tp / (((double) fp + (double) tp) + 2.220446049250313e-16); }

HD void coco_chunk_max(const CocoArgs& P, int ch, int tid, int nt) {
    const int nd = P.tot[0];
    const int base = ch * kCocoChunk, end = min(base + kCocoChunk, nd);
    for (int c = tid; c < 32; c += nt) {
        int tp = P.cpre[(size_t) ch * 64 + 2 * c], fp = P.cpre[(size_t) ch * 64 + 2 * c + 1];
        double mx = -1.0;
        for (int j = base; j < end; j++) {
            tp += (P.stp[j] >> c) & 1u;
            fp += (P.sfp[j] >> c) & 1u;
            const double p = prec(tp, fp);
            mx = p > mx ? p : mx;
        }
        P.cmax[(size_t) ch * 32 + c] = mx;
    }
}

// ---- step 4: one curve ----------------------------------------------------------------------------------------------
// the least k >= 0 with (double) k / npig >= thr, or tp_total + 1 when none is <= tp_total
HD long long least_count(double thr, int npig, int tp_total) {
    const double est = ceil(thr * (double) npig);
    long long k = !(est > 0) ? 0 : est > (double) tp_total + 1 ? (long long) tp_total + 1 : (long long) est;
    while (k > 0 && (double) (k - 1) / (double) npig >= thr) k--;
    while (k <= tp_total && !((double) k / (double) npig >= thr)) k++;
    return k;
}

HD double dmax(double x, double y) { return y > x ? y : x; }

// Curve c = a * T + t.  segmax: [nt] scratch (shared memory on the device).
HD void coco_curve(const CocoArgs& P, const int* order, int c, double* segmax, int tid, int nt) {
    const int a = c / P.T, t = c - a * P.T, R = P.R, A = P.A;
    const int nd = P.tot[0], npig = P.tot[1 + a];
    const int tp_total = P.tot[1 + 32 + 2 * c];
    if (npig == 0) {   // accumulate() skips the area: its entries keep their initial -1
        for (int r = tid; r < R; r += nt) {
            P.out.precision[((size_t) t * R + r) * A + a] = -1.0;
            P.out.scores[((size_t) t * R + r) * A + a] = -1.0;
        }
        if (tid == 0) P.out.recall[t * A + a] = -1.0;
        return;
    }
    if (tid == 0) P.out.recall[t * A + a] = nd ? (double) tp_total / (double) npig : 0.0;
    // suffix maxima of the chunk maxima (chunks past nd hold -1): thread segments, then a serial pass over the segments
    const int nch = P.n_chunks, per = (nch + nt - 1) / nt;
    double* suf = P.csuf + (size_t) c * (nch + 1);
    {
        const int b = tid * per, e = min(b + per, nch);
        double m = -1.0;
        for (int ch = b; ch < e; ch++) m = dmax(m, P.cmax[(size_t) ch * 32 + c]);
        segmax[tid] = m;
    }
    cbar();
    if (tid == 0) {
        double m = -1.0;
        for (int q = nt - 1; q >= 0; q--) { const double v = segmax[q]; segmax[q] = m; m = dmax(m, v); }
    }
    cbar();
    {
        const int b = tid * per, e = min(b + per, nch);
        double m = segmax[tid];   // the maximum of the later segments
        if (tid == nt - 1 || e == nch) suf[nch] = -1.0;
        for (int ch = e - 1; ch >= b; ch--) { m = dmax(m, P.cmax[(size_t) ch * 32 + c]); suf[ch] = m; }
    }
    cbar();
    for (int r = tid; r < R; r += nt) {
        // searchsorted(rc, recThrs[r], 'left') = the first position whose running tp count reaches k
        const long long k = least_count(P.rec[r], npig, tp_total);
        double q = 0.0, ss = 0.0;   // a position past the end: the `except: pass` leaves 0
        if (k <= tp_total && nd > 0) {
            int lo = 0, hi = nch - 1;   // the first chunk whose inclusive count reaches k (chunk 0 for k == 0)
            while (k > 0 && lo < hi) {
                const int mid = (lo + hi) / 2;
                if ((long long) P.cpre[(size_t) mid * 64 + 2 * c] + P.ccnt[(size_t) mid * 64 + 2 * c] >= k) hi = mid;
                else lo = mid + 1;
            }
            const int base = lo * kCocoChunk, end = min(base + kCocoChunk, nd);
            int tp = P.cpre[(size_t) lo * 64 + 2 * c], fp = P.cpre[(size_t) lo * 64 + 2 * c + 1];
            int i = -1;
            double mx = -1.0;
            for (int j = base; j < end; j++) {
                tp += (P.stp[j] >> c) & 1u;
                fp += (P.sfp[j] >> c) & 1u;
                if (i < 0 && tp >= k) i = j;
                if (i >= 0) mx = dmax(mx, prec(tp, fp));   // the precision envelope: max over positions >= i
            }
            if (i >= 0) {
                q = dmax(mx, suf[lo + 1]);
                ss = P.sscore[order[i]];
            }
        }
        P.out.precision[((size_t) t * R + r) * A + a] = q;
        P.out.scores[((size_t) t * R + r) * A + a] = ss;
    }
}

// ---- device kernels -------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kMatchThreads) coco_match_kernel(const CocoArgs P) {
    extern __shared__ __align__(16) unsigned char smem[];
    CocoImgWork W;
    coco_img_layout(P.max_gt, P.max_dt, P.max_det, smem, &W);
    coco_image(P, blockIdx.x, W, threadIdx.x, blockDim.x);
}

__device__ __forceinline__ unsigned digit(unsigned long long k, int shift) { return (unsigned) (k >> shift) & 255u; }

// per tile: hist[d * n_tiles + tile] = keys of digit d
__global__ void __launch_bounds__(kSortThreads) coco_sort_hist_kernel(const unsigned long long* keys, int S, int shift, unsigned* hist, int n_tiles) {
    __shared__ unsigned cnt[256];
    cnt[threadIdx.x] = 0;
    __syncthreads();
    const int base = blockIdx.x * kSortTile;
    for (int j = threadIdx.x; j < kSortTile && base + j < S; j += kSortThreads) atomicAdd(&cnt[digit(keys[base + j], shift)], 1u);
    __syncthreads();
    hist[(size_t) threadIdx.x * n_tiles + blockIdx.x] = cnt[threadIdx.x];
}

// exclusive scan of hist [256 * n_tiles] in place, one block: each thread a contiguous segment
__global__ void __launch_bounds__(kScanThreads) coco_sort_scan_kernel(unsigned* hist, int n) {
    typedef cub::BlockScan<unsigned, kScanThreads> Scan;
    __shared__ typename Scan::TempStorage tmp;
    const int per = (n + kScanThreads - 1) / kScanThreads;
    const int b = threadIdx.x * per, e = min(b + per, n);
    unsigned s = 0;
    for (int j = b; j < e; j++) s += hist[j];
    unsigned pre;
    Scan(tmp).ExclusiveSum(s, pre);
    for (int j = b; j < e; j++) { const unsigned v = hist[j]; hist[j] = pre; pre += v; }
}

// stable scatter of one tile by the digit at `shift`
__global__ void __launch_bounds__(kSortThreads) coco_sort_scatter_kernel(const unsigned long long* kin, const int* vin, unsigned long long* kout,
                                                                         int* vout, int S, int shift, const unsigned* hist, int n_tiles) {
    typedef cub::BlockRadixSort<unsigned long long, kSortThreads, kSortItems, int> Sort;
    __shared__ typename Sort::TempStorage tmp;
    __shared__ unsigned start[256], goff[256];
    const int base = blockIdx.x * kSortTile, len = min(kSortTile, S - base);
    unsigned long long k[kSortItems];
    int v[kSortItems];
    for (int q = 0; q < kSortItems; q++) {
        const int j = threadIdx.x * kSortItems + q;
        k[q] = j < len ? kin[base + j] : kPadKey;
        v[q] = j < len ? vin[base + j] : 0;
    }
    start[threadIdx.x] = 0;
    goff[threadIdx.x] = hist[(size_t) threadIdx.x * n_tiles + blockIdx.x];
    __syncthreads();
    for (int q = 0; q < kSortItems; q++)
        if (threadIdx.x * kSortItems + q < len) atomicAdd(&start[digit(k[q], shift)], 1u);
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned s = 0;
        for (int d = 0; d < 256; d++) { const unsigned c = start[d]; start[d] = s; s += c; }
    }
    Sort(tmp).Sort(k, v, shift, shift + 8);   // stable: equal digits keep their tile order; the padding sorts last
    __syncthreads();
    for (int q = 0; q < kSortItems; q++) {
        const int pos = threadIdx.x * kSortItems + q;
        if (pos >= len) continue;
        const unsigned d = digit(k[q], shift);
        const unsigned o = goff[d] + (unsigned) pos - start[d];
        kout[o] = k[q];
        vout[o] = v[q];
    }
}

__global__ void __launch_bounds__(kChunkThreads) coco_chunk_counts_kernel(const CocoArgs P, const int* order) {
    __shared__ unsigned stage[2 * kCocoChunk];
    coco_chunk_counts(P, order, blockIdx.x, stage, threadIdx.x, blockDim.x);
}

// totals and the exclusive prefix of the chunk counts, one block: column u = 2c + kind, 16 segments of chunks each
HD void coco_totals(const CocoArgs& P, int tid, int nt, int* seg_sum /* [16][64] */) {
    const int nseg = nt >= 1024 ? 16 : 1;
    const int per = (P.n_chunks + nseg - 1) / nseg;
    for (int w = tid; w < nseg * 64; w += nt) {
        const int sg = w / 64, u = w - sg * 64;
        const int b = sg * per, e = min(b + per, P.n_chunks);
        int s = 0;
        for (int ch = b; ch < e; ch++) s += P.ccnt[(size_t) ch * 64 + u];
        seg_sum[w] = s;
    }
    cbar();
    for (int w = tid; w < nseg * 64; w += nt) {
        const int sg = w / 64, u = w - sg * 64;
        int s = 0;
        for (int q = 0; q < sg; q++) s += seg_sum[q * 64 + u];
        const int b = sg * per, e = min(b + per, P.n_chunks);
        for (int ch = b; ch < e; ch++) { P.cpre[(size_t) ch * 64 + u] = s; s += P.ccnt[(size_t) ch * 64 + u]; }
        if (sg == nseg - 1) P.tot[1 + 32 + u] = s;
    }
    if (tid == 0) {
        long long nd = 0;
        for (int i = 0; i < P.n_img; i++) nd += P.kept[i];
        P.tot[0] = (int) nd;
    }
    for (int a = tid; a < P.A; a += nt) {
        int s = 0;
        for (int i = 0; i < P.n_img; i++) s += P.npig_img[(size_t) i * P.A + a];
        P.tot[1 + a] = s;
    }
}
__global__ void __launch_bounds__(kScanThreads) coco_totals_kernel(const CocoArgs P) {
    __shared__ int seg[16 * 64];
    coco_totals(P, threadIdx.x, blockDim.x, seg);
}
__global__ void __launch_bounds__(kChunkThreads) coco_chunk_max_kernel(const CocoArgs P) {
    coco_chunk_max(P, blockIdx.x, threadIdx.x, blockDim.x);
}
__global__ void __launch_bounds__(kCurveThreads) coco_curve_kernel(const CocoArgs P, const int* order) {
    __shared__ double segmax[kCurveThreads];
    coco_curve(P, order, blockIdx.x, segmax, threadIdx.x, blockDim.x);
}

// ---- launchers ------------------------------------------------------------------------------------------------------
cudaError_t configure_coco_eval() {
    return cudaFuncSetAttribute(coco_match_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) kCocoSmemMax);
}
size_t coco_img_smem_bytes(int max_gt, int max_dt, int max_det) { return coco_img_layout(max_gt, max_dt, max_det, nullptr, nullptr); }
int coco_eval_launches() { return 1 + 3 * kSortPasses + 4; }

static CocoArgs coco_args(const ekp_coco_gt& gt, int max_gt, const ekp_coco_dt& dt, int max_dt, int n_img, int max_det,
                          const double* iou, int T, const double* rec, int R, const double* area, int A, void* ws,
                          const ekp_coco_eval_out& out) {
    CocoArgs P;
    coco_ws_layout(n_img, max_det, A, static_cast<unsigned char*>(ws), &P);
    P.gt = gt; P.dt = dt; P.max_gt = max_gt; P.max_dt = max_dt; P.n_img = n_img; P.max_det = max_det;
    P.T = T; P.R = R; P.A = A; P.iou = iou; P.rec = rec; P.area = area; P.out = out;
    oks_vars(P.var);
    return P;
}

cudaError_t launch_coco_eval(const ekp_coco_gt& gt, int max_gt, const ekp_coco_dt& dt, int max_dt, int n_img, int max_det,
                             const double* iou, int T, const double* rec, int R, const double* area, int A, void* ws,
                             const ekp_coco_eval_out& out, cudaStream_t st) {
    const CocoArgs P = coco_args(gt, max_gt, dt, max_dt, n_img, max_det, iou, T, rec, R, area, A, ws, out);
    coco_match_kernel<<<n_img, kMatchThreads, coco_img_smem_bytes(max_gt, max_dt, max_det), st>>>(P);
    for (int p = 0; p < kSortPasses; p++) {
        const int in = p & 1;
        coco_sort_hist_kernel<<<P.n_tiles, kSortThreads, 0, st>>>(P.key[in], P.S, 8 * p, P.hist, P.n_tiles);
        coco_sort_scan_kernel<<<1, kScanThreads, 0, st>>>(P.hist, 256 * P.n_tiles);
        coco_sort_scatter_kernel<<<P.n_tiles, kSortThreads, 0, st>>>(P.key[in], P.val[in], P.key[in ^ 1], P.val[in ^ 1], P.S,
                                                                     8 * p, P.hist, P.n_tiles);
    }
    const int* order = P.val[kSortPasses & 1];
    coco_chunk_counts_kernel<<<P.n_chunks, kChunkThreads, 0, st>>>(P, order);
    coco_totals_kernel<<<1, kScanThreads, 0, st>>>(P);
    coco_chunk_max_kernel<<<P.n_chunks, kChunkThreads, 0, st>>>(P);
    coco_curve_kernel<<<A * T, kCurveThreads, 0, st>>>(P, order);
    return cudaGetLastError();
}

void debug_coco_eval_host(const ekp_coco_gt& gt, int max_gt, const ekp_coco_dt& dt, int max_dt, int n_img, int max_det,
                          const double* iou, int T, const double* rec, int R, const double* area, int A,
                          const ekp_coco_eval_out& out) {
    std::vector<double> ws(coco_eval_ws_bytes(n_img, max_det, A) / sizeof(double) + 1);
    const CocoArgs P = coco_args(gt, max_gt, dt, max_dt, n_img, max_det, iou, T, rec, R, area, A, ws.data(), out);
    std::vector<double> img(coco_img_smem_bytes(max_gt, max_dt, max_det) / sizeof(double) + 1);
    CocoImgWork W;
    coco_img_layout(max_gt, max_dt, max_det, reinterpret_cast<unsigned char*>(img.data()), &W);
    for (int i = 0; i < n_img; i++) coco_image(P, i, W, 0, 1);
    std::vector<int> order(P.S);
    for (int s = 0; s < P.S; s++) order[s] = s;
    std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return P.key[0][x] < P.key[0][y]; });
    std::vector<unsigned> stage(2 * kCocoChunk);
    for (int ch = 0; ch < P.n_chunks; ch++) coco_chunk_counts(P, order.data(), ch, stage.data(), 0, 1);
    std::vector<int> seg(64);
    coco_totals(P, 0, 1, seg.data());
    for (int ch = 0; ch < P.n_chunks; ch++) coco_chunk_max(P, ch, 0, 1);
    double segmax[1];
    for (int c = 0; c < A * T; c++) coco_curve(P, order.data(), c, segmax, 0, 1);
}

}  // namespace ekp
