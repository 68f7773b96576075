/* ekpose_b200.h -- C ABI of libekpose_b200.so: the B200 (sm_100a) implementation of
 * torch_ekpose's PAF post-processing hot path.
 *
 * Two surfaces are exported, both plain C (pointers and sizes only, no torch / C++ types):
 *
 * 1. The reference's own operator surface, so the library is a drop-in for the SWIG module
 *    `lib.pafprocess.pafprocess`:
 *        process_paf / get_num_humans / get_part_cid / get_score /
 *        get_part_x / get_part_y / get_part_score
 *    replace, name for name and argument for argument, the functions declared at
 *    /root/reference/lib/pafprocess/pafprocess.h:53-59 (defined pafprocess.cpp:22-218, bound
 *    to Python by pafprocess.i:14-15).  HOST pointers in, results held process-globally until
 *    the next process_paf call, exactly like the reference (pafprocess.cpp:12-13).  The work
 *    (stages 4-5) runs on the GPU; there is no CPU fallback: without a CUDA device
 *    process_paf returns EKP_ERR_CUDA and ekp_last_error() says why.
 *
 * 2. A handle-based batched API on DEVICE (or pinned host) tensors that also covers the
 *    Python-side preprocessing of the reference (lib/utils/paf_to_pose.py: find_peaks :26-36,
 *    NMS :60-133, the upsampling of paf_to_pose_cpp :356-359) as CUDA stages 1-3, so a whole
 *    batch goes from the network's stride-8 outputs to people in one call.  The people come back as host tables
 *    (ekp_results, ekp_results_humans: these wait for the run) or into caller-owned device buffers, ordered on a
 *    stream with no host wait (ekp_results_device, ekp_results_device_peaks).  A caller that reads them only on the
 *    device can also skip each batch's copy of the result records to the host (ekp_set_host_copy), and give its people
 *    stable ids across video frames on the device (ekp_track_humans), and smooth their keypoints per id
 *    (ekp_smooth_humans).
 *
 * All functions return EKP_OK (0) or a negative ekp_status; ekp_last_error() returns a
 * thread-local human-readable message for the last failure.  Nothing aborts.
 */
#ifndef EKPOSE_B200_H
#define EKPOSE_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EKP_NUM_PART 18      /* pafprocess.h:11 NUM_PART */
#define EKP_NUM_LIMB 19      /* pafprocess.h:15 COCOPAIRS_SIZE */
#define EKP_HEAT_CH 19       /* 18 parts + background (lib/network/vgg2016.py:105) */
#define EKP_PAF_CH 38        /* 19 limbs x (x, y) */
#define EKP_UP 8             /* lib/config/default.py:17 MODEL.DOWNSAMPLE */
#define EKP_SUBSET_COLS 20   /* 18 cids + score sum + part count (pafprocess.cpp:174-181) */

typedef enum ekp_status {
    EKP_OK = 0,
    EKP_ERR_ARG = -1,       /* bad dimensions / null pointer / part id outside [0,18) / non-finite input */
    EKP_ERR_CUDA = -2,      /* CUDA runtime error or no device */
    EKP_ERR_CAPACITY = -3,  /* a fixed-capacity buffer overflowed (see ekp_results `overflow`) */
    EKP_ERR_STATE = -4      /* results requested before any run, etc. */
} ekp_status;

typedef enum ekp_layout { EKP_LAYOUT_NCHW = 0, EKP_LAYOUT_NHWC = 1 } ekp_layout;

/* element type of the heat / PAF inputs of the *_typed entry points.  16-bit maps (what the network returns under
 * torch.autocast) are widened to float32 on the device (exact: every finite value, +-0, subnormals and +-inf; a NaN
 * stays a NaN) and then take the float32 path, so the results equal those of the float32 maps x.float(). */
typedef enum ekp_dtype { EKP_DTYPE_F32 = 0, EKP_DTYPE_BF16 = 1, EKP_DTYPE_F16 = 2 } ekp_dtype;

/* which peak front-end runs as stages 1-3 */
typedef enum ekp_frontend {
    EKP_FRONTEND_DENSE = 0,     /* bilinear x8 -> Gaussian sigma 3 -> 3x3 max NMS (BASELINE.json north_star) */
    EKP_FRONTEND_REFERENCE = 1, /* the reference's NMS(): stride-8 cross NMS + bicubic patch refinement */
    EKP_FRONTEND_REFERENCE_COARSE = 2, /* NMS(bool_refine_center=False) / find_peaks (paf_to_pose.py:26-36, :119-122): the
                                       * stride-8 maxima themselves, reported at (8c + 3) = (int) compute_resized_coords(c, 8)
                                       * (:39-57, truncated like pafprocess.cpp:30-31) with the heat value as score */
    EKP_FRONTEND_REFERENCE_GAUSS = 3   /* NMS(bool_gaussian_filt=True), paf_to_pose.py:111-112: as REFERENCE, with
                                       * scipy.ndimage.gaussian_filter(sigma=3) applied to every upsampled patch before the
                                       * arg-max (no caller in the reference enables it; bit-exact against scipy) */
} ekp_frontend;

/* per-image overflow bits reported by ekp_results */
#define EKP_OVF_PEAKS 1u       /* more peaks than max_peaks */
#define EKP_OVF_PART 2u        /* more than max_part peaks of one part */
#define EKP_OVF_CANDIDATES 4u  /* more than max_cand passing candidates on one limb */
#define EKP_OVF_HUMANS 8u      /* more subset rows than max_humans */
#define EKP_OVF_BADPEAK 16u    /* a peak had part id outside [0,18) or coordinates outside the PAF map */

/* Default per-image capacities of a context made by ekp_create; ekp_create_ex sets them per context.  The
 * reference keeps unbounded std::vectors (pafprocess.cpp:24, :47-49); here a scene that exceeds a capacity is
 * REPORTED (EKP_OVF_*, EKP_ERR_CAPACITY), and the caller re-creates the context with larger ones (the Python
 * host layer and the process_paf surface grow and retry by themselves). */
#define EKP_MAX_PART 256       /* peaks of one part per image */
#define EKP_MAX_CAND 2048      /* candidates that pass both criteria, per limb per image */
/* hard limits of ekp_create_ex */
#define EKP_LIMIT_PEAKS 16384
#define EKP_LIMIT_HUMANS 1024
#define EKP_LIMIT_PART 1024
#define EKP_LIMIT_CAND 8192

/* one row of the part-sorted peak table (pafprocess.h:26-31 `Peak`) */
typedef struct ekp_peak {
    int x;
    int y;
    float score;
    int id;
} ekp_peak;

typedef struct ekp_ctx ekp_ctx;

/* Create a context on CUDA device `device` with fixed-capacity work buffers:
 * up to max_batch images per call, stride-8 maps up to max_h x max_w, at most max_peaks peaks
 * and max_humans subset rows per image.  One context = one stream of work; contexts are
 * independent, so one host thread per GPU can drive its own. */
int ekp_create(ekp_ctx **out, int device, int max_batch, int max_h, int max_w, int max_peaks, int max_humans);
/* Same with the two remaining capacities explicit (0 = the defaults above): max_part peaks of one part and
 * max_cand passing candidates of one limb, per image.  Smaller values leave more shared memory per block
 * (more resident blocks in stage 4), larger ones (up to EKP_LIMIT_*) take scenes the defaults report as overflow. */
int ekp_create_ex(ekp_ctx **out, int device, int max_batch, int max_h, int max_w, int max_peaks, int max_humans,
                  int max_part, int max_cand);
void ekp_destroy(ekp_ctx *ctx);
const char *ekp_last_error(void);
const char *ekp_version(void);

/* Stages 1-5 on DEVICE tensors (asynchronous on `stream`, a cudaStream_t passed as void*).
 *   heat  float32 [n,19,h,w] (NCHW) or [n,h,w,19] (NHWC): the network's heat-map output
 *   paf   float32 [n,38,h,w] / [n,h,w,38]
 *   thr_heat  lib/config/default.py:23 TEST.THRESH_HEATMAP (0.15)
 *   heat_mat / paf_mat  optional DEVICE outputs float32 [n,8h,8w,19] / [n,8h,8w,38]: the full
 *       resolution operator-surface tensors the reference hands to process_paf
 *       (paf_to_pose.py:356-360).  DENSE front-end: bilinear x8 (paf_mat is then also what
 *       stage 4 samples); REFERENCE front-end: nearest x8.  Pass NULL to skip materialising;
 *       stage 4 then computes the identical sample values from the stride-8 PAF.
 *       Both must be 16-byte aligned (they are written by the TMA engine in 16-byte units); heat / paf need
 *       only their natural 4-byte alignment.
 * Replaces paf_to_pose_cpp lines 346-360 (NMS + upsample + process_paf) for a whole batch. */
int ekp_postprocess(ekp_ctx *ctx, const float *heat, const float *paf, int n, int h, int w, int layout,
                    float thr_heat, int frontend, float *heat_mat, float *paf_mat, void *stream);

/* Same, but heat / paf are HOST buffers (ideally pinned): copies them to the context's device
 * buffers on `stream` first.  materialize != 0 writes heat_mat / paf_mat into context-owned
 * device buffers (they are not copied back). */
int ekp_postprocess_host(ekp_ctx *ctx, const float *heat_host, const float *paf_host, int n, int h, int w,
                         int layout, float thr_heat, int frontend, int materialize, void *stream);

/* ekp_postprocess / ekp_postprocess_host for inputs of element type `dtype` (ekp_dtype).  EKP_DTYPE_F32 is exactly the
 * two calls above.  EKP_DTYPE_BF16 / EKP_DTYPE_F16: heat / paf hold 16-bit values in the same shapes and layouts and
 * need 2-byte alignment; one kernel widens both to float32 into a context-owned device block (allocated on first use,
 * max_batch x max_h x max_w x 57 floats), then the float32 kernels run on it.  heat_mat / paf_mat stay float32.
 * The host variant copies the 16-bit buffers (half the bytes of float32) into a second context-owned 16-bit device
 * block first: ONE copy when heat is directly followed by paf in host memory, as for float32.  The widening kernel
 * counts in ekp_kernel_launches, its time in stage [0] of ekp_stage_times, and it is part of the batch's CUDA graph.
 * An unknown dtype or a 16-bit pointer that is not 2-byte aligned returns EKP_ERR_ARG. */
int ekp_postprocess_typed(ekp_ctx *ctx, const void *heat, const void *paf, int dtype, int n, int h, int w, int layout,
                          float thr_heat, int frontend, float *heat_mat, float *paf_mat, void *stream);
int ekp_postprocess_host_typed(ekp_ctx *ctx, const void *heat_host, const void *paf_host, int dtype, int n, int h,
                               int w, int layout, float thr_heat, int frontend, int materialize, void *stream);

/* Stages 4-5 only, DEVICE inputs: per image a peak list in the reference's format
 * float32 [n, peaks_stride, 5] rows (x, y, score, <ignored>, part) (pafprocess.cpp:26-36) with
 * n_peaks[i] valid rows, and the full-resolution PAF tensor float32 [n, H, W, C] the reference
 * indexes (pafprocess.cpp:8).  h1 is heat_mat.shape[0], the only use of heat_mat (:83). */
int ekp_process_paf_dev(ekp_ctx *ctx, const float *peaks, const int *n_peaks, int peaks_stride, int n, int h1,
                        const float *paf_mat, int H, int W, int C, void *stream);

/* Wait for the last run and copy its results out (any pointer may be NULL):
 *   num_humans [n]                      people per image (pafprocess.cpp:196-198)
 *   subset     [n, max_humans, 20]      rows as the reference keeps them (:127-191), float32
 *   n_peaks    [n]                      peaks per image
 *   peaks_line [n, max_peaks]           part-sorted peak table (:38-43)
 *   overflow   [n]                      EKP_OVF_* bits
 * Returns EKP_ERR_CAPACITY if any image overflowed (outputs are still written). */
int ekp_results(ekp_ctx *ctx, int *num_humans, float *subset, int *n_peaks, ekp_peak *peaks_line,
                unsigned *overflow);

/* Vectorised form of the getter loop of paf_to_pose_cpp (:361-377): per human and part the
 * peak (x, y, score, id = cid or -1 when the part is absent) as ekp_peak [n, max_humans, 18],
 * i.e. get_part_cid / get_part_x / get_part_y / get_part_score in one table, and the human score
 * float32 [n, max_humans] = subset[18] / subset[19] (get_score, pafprocess.cpp:204-206). */
int ekp_results_humans(ekp_ctx *ctx, int *num_humans, ekp_peak *parts, float *scores, unsigned *overflow);

/* ---- results on the device ---------------------------------------------------------------------
 * The tables of ekp_results / ekp_results_humans written into caller-owned DEVICE buffers instead of host arrays, so a
 * caller that keeps the people on the GPU (a tracker, a second model, crops) neither waits for the run nor copies them
 * back.  Every pointer is a device pointer, 4-byte aligned, and may be NULL (that table is not written). */
typedef struct ekp_device_results {
    int *num_humans;      /* [n]                     people per image */
    unsigned *overflow;   /* [n]                     EKP_OVF_* bits */
    int *n_peaks;         /* [n]                     peaks per image */
    float *subset;        /* [n, max_humans, 20]     as ekp_results */
    ekp_peak *parts;      /* [n, max_humans, 18]     as ekp_results_humans */
    float *scores;        /* [n, max_humans]         as ekp_results_humans */
} ekp_device_results;
/* Writes the last run's tables into `out` for its n = ekp_last_batch(ctx) images.  Rows from num_humans[i] up to
 * max_humans are written as zero bytes, so each table copied to the host equals the host call's byte for byte, padding
 * included.  One kernel launch (counted in ekp_kernel_launches; not part of the batch's CUDA graph), asynchronous on
 * `stream` and ordered like ekp_draw_humans: after the run (an export on another stream waits for it), and before the
 * context's next run on any stream.  It never waits on the host and never allocates.  Works after every batched entry
 * point (ekp_postprocess*, ekp_postprocess_host*, ekp_process_paf_dev).
 * Overflow does not fail the call (nothing is known about it at call time): the bits land in `overflow`, and the caller
 * checks them.  EKP_ERR_STATE before any run; EKP_ERR_ARG for a NULL context or out, n != ekp_last_batch(ctx) or a
 * pointer that is not 4-byte aligned.  All pointers NULL: EKP_OK, nothing is launched. */
int ekp_results_device(ekp_ctx *ctx, int n, const ekp_device_results *out, void *stream);

/* The part-sorted peak table of the last run in caller-owned DEVICE buffers (4-byte aligned; NULL: not written):
 * the device counterpart of ekp_results' n_peaks / peaks_line and ekp_results_parts. */
typedef struct ekp_device_peaks {
    int *n_peaks;         /* [n]                     peaks per image */
    ekp_peak *peaks;      /* [n, max_peaks]          part-sorted peak table, as ekp_results' peaks_line */
    int *part_off;        /* [n, 19]                 as ekp_results_parts */
} ekp_device_peaks;
/* Writes the last run's peak tables into `out`: one kernel launch, ordered and checked exactly like ekp_results_device
 * (same error codes; all pointers NULL: EKP_OK, nothing is launched).  Rows from min(n_peaks[i], max_peaks) up to
 * max_peaks are written as zero bytes, so the table copied to the host equals ekp_results' peaks_line padding
 * included. */
int ekp_results_device_peaks(ekp_ctx *ctx, int n, const ekp_device_peaks *out, void *stream);

/* Whether batches end with the device-to-host copy of their result records.  enable != 0 (the default): every batch
 * of ekp_postprocess*, ekp_postprocess_host* and ekp_process_paf_dev ends with one copy of max_humans-sized records
 * into pinned host memory, which the host readers (ekp_results, ekp_results_humans) then read without touching the
 * device.  enable == 0: batches submitted from now on leave the records on the device only.  That suits a caller who
 * reads results only on the device (ekp_results_device*, ekp_draw_humans) and saves the copy on every batch (about
 * 0.75 MB for 64 images at max_humans 32).  The host readers still work after such a run: the first of them waits for
 * it and downloads its records once.  The mode is recorded with each run, so changing it does not affect a run
 * already submitted, and each mode replays its own CUDA graph.  The process_paf surface is not affected. */
int ekp_set_host_copy(ekp_ctx *ctx, int enable);

/* ---- tracking: stable person ids across video frames ----------------------------------------------------------------
 * Gives every person of a frame the id of the same person in earlier frames of its sequence, from the device human
 * tables (ekp_results_device's num_humans and parts), so a video caller keeps the people on the GPU from frame to id.
 * A call takes the tables of n images and n_seq sequences (n % n_seq == 0, F = n / n_seq): image i is frame i % F of
 * sequence i / F.  n_seq = 1 is a batch of consecutive frames of one video, F = 1 is n_seq cameras with one frame each.
 * Each sequence keeps its own tracks, frame counter and next id (ids start at 0 and grow by 1 per new track) in `state`,
 * across calls.  The people of image i are rows 0 .. min(num_humans[i], max_humans) - 1 of parts [n, max_humans, 18]
 * (overflow or not: the table is tracked as it stands).
 *   similarity  COCO's OKS in float64 against the track's last pose: keypoint j = reference part ORDER_COCO[j]
 *               (torch_ekpose_b200/coco.py; the neck is not used), pycocotools' sigmas / 10 and vars = (2 sigma)^2,
 *               area = the integer (xmax - xmin + 1) * (ymax - ymin + 1) of the track's present keypoints, and over the m
 *               keypoints present in both, in order of j, e_j = d2_j / var_j / area / 2 (d2_j = dx*dx + dy*dy, exact):
 *               sim = sum of exp(-e_j) / m, or 0 when m == 0.
 *   matching    per frame, the pairs (person, live track) with sim >= (double) min_oks, in descending sim, then
 *               ascending track id, then ascending row; a pair is accepted when neither side is taken.  A matched person
 *               gets its track's id, and the track its whole pose.  Unmatched people open new tracks in row order.
 *   age         a track last matched at frame f0 can be matched at frames f0 + 1 .. f0 + max_age + 1, then is dropped.
 *   capacity    a new track that finds all max_tracks slots live takes the slot of the track with the smallest last
 *               match frame, then the smallest id, among those neither matched nor opened in this frame.
 * ids int32 [n, max_humans] gets each row's track id, and -1 from row num_humans[i] on.
 * Every pointer is a caller-owned DEVICE pointer: the tables and ids 4-byte aligned, the state 8-byte aligned.  The
 * state's layout is private; its size depends only on (n_seq, max_tracks), so it outlives any context (a context
 * re-created with larger capacities keeps tracking on the same state).  It holds the track poses and, per sequence, a
 * max_tracks x max_tracks scratch of similarities for frames whose pairs do not fit shared memory.  Poses are kept in
 * the map pixels of the runs that produced them: feeding one sequence runs of a different map size is the caller's
 * error.  Frame counters are 32-bit.
 * ekp_track_humans is one kernel launch (one block per sequence, counted in ekp_kernel_launches, not part of any batch
 * graph), asynchronous on `stream`; it never waits on the host and never allocates.  The context only supplies the
 * device and the error reporting: the call reads the caller's tables, not the context's records, so it composes with
 * ekp_results_device on the same stream, and ordering across streams is the caller's.  EKP_ERR_ARG for a NULL pointer,
 * n < 1 or n % n_seq != 0, max_humans outside [1, max_tracks], max_tracks outside [1, EKP_LIMIT_TRACKS], max_age < 0, a
 * negative or non-finite min_oks, or a misaligned pointer. */
#define EKP_LIMIT_TRACKS 512   /* slots of one sequence: at max_humans = max_tracks = 512 the per-block working set
                                * (tracks, the frame's people, lists) takes 172,192 of the 232,448 bytes of shared memory
                                * of one block, and the rest holds the similarity matrix */
/* Bytes of a state for n_seq sequences of up to max_tracks tracks; 0 when n_seq < 1 or max_tracks is outside
 * [1, EKP_LIMIT_TRACKS].  long long rather than size_t: every function of this header returns int, float, long long,
 * void or a pointer, the set tests/test_abi.py parses to check the header against the library and its Python binding;
 * the value is a non-negative byte count. */
long long ekp_track_state_bytes(int n_seq, int max_tracks);
/* Clears a state asynchronously on `stream` (cudaMemsetAsync): no tracks, frame 0, next id 0 in every sequence. */
int ekp_track_reset(ekp_ctx *ctx, void *state, int n_seq, int max_tracks, void *stream);
int ekp_track_humans(ekp_ctx *ctx, const int *num_humans, const ekp_peak *parts, int n, int max_humans, void *state,
                     int n_seq, int max_tracks, float min_oks, int max_age, int *ids, void *stream);
/* Test hook for ekp_track_humans: the same code, run serially on the CPU on HOST buffers (and a host state), with the same
 * arguments and checks.  It is not a CPU path of the tracker. */
int ekp_debug_track_host(const int *num_humans, const ekp_peak *parts, int n, int max_humans, void *state, int n_seq,
                         int max_tracks, float min_oks, int max_age, int *ids);

/* ---- smoothing: One Euro filtered keypoints across video frames, per track --------------------------------------------
 * Smooths the people's keypoints from frame to frame with a One Euro filter (Casiez, Roussel, Vogel, CHI 2012) per track
 * id, part and axis, on the device human tables (ekp_results_device's num_humans and parts) and the ids ekp_track_humans
 * wrote for them.  Both front-ends report integer map pixels, so a still person's keypoints jump by a pixel or more
 * between frames; the filter removes that jitter at low speed and follows fast motion with little lag.
 * A call takes n images and n_seq sequences as ekp_track_humans does (n % n_seq == 0, F = n / n_seq, image i is frame
 * i % F of sequence i / F).  Each sequence keeps its own frame counter and up to max_tracks entries, one per track id,
 * in `state`, across calls.  An entry holds, per reference part (all 18, the neck included, in part order) and axis, the
 * filter values xh, dxh and the frame of the part's last sample.  For row p < min(num_humans[i], max_humans) with
 * id = ids[i][p]:
 *   id < 0      the row is passed through: its output is its raw coordinates, and it touches no entry.
 *   lookup      the row uses the entry of its id.  Without one, it opens one: in a free entry if there is one, else in
 *               the entry with the smallest (last_seen, id) among those not seen in this frame.  A frame first resolves
 *               every row whose id already has an entry, and only then opens entries, in row order: a birth never
 *               evicts an entry a later row of the same frame uses.
 *   expiry      an entry last seen at frame f0 is dropped at frame f0 + max_age + 2 (the tracker's rule).
 *   duplicates  ids within a frame must be distinct; duplicates give unspecified coordinates, never an out-of-bounds
 *               access.
 * With the (n_seq, max_tracks, max_age) of the ekp_track_humans call that produced the ids, the live entries are exactly
 * the tracker's live tracks, so a filter restarts only when its track is born.
 * Per present part (parts[..].id >= 0) and axis, with the raw value x = (double) coordinate at frame f, a part's first
 * sample in its entry (an opened entry has none) sets xh = x, dxh = 0; every later one, with g = f - (frame of the
 * part's last sample) and pi the double nearest pi, does in this order, each an IEEE float64 operation, uncontracted:
 *     te = (double) g / fps            tau_d = 1.0 / ((2.0 * pi) * d_cutoff)     a_d = 1.0 / (1.0 + tau_d / te)
 *     dx = (x - xh) / te               dxh = a_d * dx + (1.0 - a_d) * dxh
 *     c = min_cutoff + beta * fabs(dxh)
 *     tau = 1.0 / ((2.0 * pi) * c)     a = 1.0 / (1.0 + tau / te)                xh = a * x + (1.0 - a) * xh
 * An absent part leaves its values as they are: its next sample uses the real gap g.
 * xy float32 [n, max_humans, 18, 2] gets (float) xh, rounded to nearest, for every present part of a row with an entry,
 * the raw coordinates for the present parts of passed-through rows, and 0.0f for absent parts and rows from num_humans[i]
 * on, so a dirty buffer is fully overwritten; presence stays readable from parts[..., 3].  Coordinates are map pixels
 * like the tables' (frame rates, cutoffs and beta are per frame of fps and per pixel accordingly).
 * Every pointer is a caller-owned DEVICE pointer: the tables, ids and xy 4-byte aligned, the state 8-byte aligned.  The
 * state's layout is private; its size depends only on (n_seq, max_tracks), so it outlives any context.  Frame counters
 * are 32-bit.  ekp_smooth_humans is one kernel launch (one block per sequence, counted in ekp_kernel_launches),
 * asynchronous on `stream`; it never waits on the host and never allocates.  The context only supplies the device and
 * the error reporting.  EKP_ERR_ARG for a NULL pointer, n < 1 or n % n_seq != 0, max_humans outside [1, max_tracks],
 * max_tracks outside [1, EKP_LIMIT_TRACKS], max_age < 0, an fps, min_cutoff or d_cutoff that is not finite and
 * positive, a beta that is not finite and non-negative, or a misaligned pointer. */
/* Bytes of a state for n_seq sequences of up to max_tracks entries (16 per sequence and 728 per entry); 0 when n_seq < 1 or max_tracks is
 * outside [1, EKP_LIMIT_TRACKS]. */
long long ekp_smooth_state_bytes(int n_seq, int max_tracks);
/* Clears a state asynchronously on `stream` (cudaMemsetAsync): no entries, frame 0 in every sequence. */
int ekp_smooth_reset(ekp_ctx *ctx, void *state, int n_seq, int max_tracks, void *stream);
int ekp_smooth_humans(ekp_ctx *ctx, const int *num_humans, const ekp_peak *parts, const int *ids, int n, int max_humans,
                      void *state, int n_seq, int max_tracks, int max_age, double fps, double min_cutoff, double beta,
                      double d_cutoff, float *xy, void *stream);
/* Test hook for ekp_smooth_humans: the same code, run serially on the CPU on HOST buffers (and a host state), with the
 * same arguments and checks.  It is not a CPU path of the smoother. */
int ekp_debug_smooth_host(const int *num_humans, const ekp_peak *parts, const int *ids, int n, int max_humans, void *state,
                          int n_seq, int max_tracks, int max_age, double fps, double min_cutoff, double beta, double d_cutoff,
                          float *xy);

/* ---- COCO keypoint evaluation: pycocotools' COCOeval(iouType='keypoints') on the device ------------------------------
 * Scores detected people against COCO person-keypoint ground truth, one category, and writes accumulate()'s precision,
 * recall and scores arrays, equal bit for bit to pycocotools' (float64 throughout).  Inputs are padded per-image tables
 * of n_img images: image order is row order (the Python packers sort by image id, as pycocotools' np.unique does), and
 * within an image rows are in annotation order (gt) or result-list order (dt); counts are clamped to [0, max_gt] /
 * [0, max_dt].  The rules, as pycocotools states them:
 *   dt area      (loadRes) over all 17 keypoints, absent (0, 0, 0) triples included: (max x - min x) * (max y - min y).
 *   gt ignore    (_prepare) iscrowd or num_keypoints == 0, packed into `ignore` by the caller.
 *   dt order     a stable sort by descending score, truncated to max_det; -0.0 and +0.0 compare equal.
 *   OKS          (computeOks) vars = (2 sigma)^2 with pycocotools' sigmas; k1 = gt keypoints with v > 0.  k1 > 0:
 *                dx = xd - xg over those keypoints; k1 == 0: dx = max(0, x0 - xd) + max(0, xd - x1) with x0 = bx - bw,
 *                x1 = bx + 2 bw from the gt bbox (likewise y), over all 17.  e = (dx^2 + dy^2) / vars / (area + 2^-52) / 2,
 *                oks = sum(exp(-e)) / len(e), the sum in numpy's pairwise order (sequential below 8 terms, else eight
 *                accumulators over the multiple-of-8 prefix, ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)), then the rest).
 *   matching     (evaluateImg) per image, area range a = [lo, hi] and threshold t: gts stable-sorted by
 *                _ignore = ignore or area outside [lo, hi]; each dt in order starts from iou = min(t, 1 - 1e-10) and
 *                scans the gts, skipping one already matched at t unless it is a crowd, stopping at the first ignored gt
 *                once its match is a non-ignored one, skipping oks < iou, else taking iou = oks and that gt (so among equal
 *                OKS the last gt wins).  A matched dt is ignored when its gt is; an unmatched one when its own area is
 *                outside [lo, hi].
 *   accumulate   all kept dts of all images, concatenated in image order and stable-sorted by descending score;
 *                npig = non-ignored gts of area a (0: that area's entries stay -1); tp / fp running counts in float64,
 *                rc = tp / npig, pr = tp / ((fp + tp) + 2^-52), pr replaced by its running maximum from the end;
 *                i = searchsorted(rc, recThrs[r], 'left'), precision = pr[i] and scores = the i-th sorted score, both 0
 *                when i is past the end; recall = rc[-1], or 0 with no detections.
 * The thresholds are inputs: iou_thrs [T], rec_thrs [R] and area_rng [A][2] (pycocotools' np.linspace values and
 * [[0, 1e10], [32^2, 96^2], [96^2, 1e10]] for its keypoint defaults).  Non-finite inputs give unspecified numbers, never
 * an out-of-bounds access.  Every pointer is a caller-owned DEVICE pointer (host pointers for the test hook), 8-byte
 * aligned; the tables are float64 where pycocotools keeps floats, int32 otherwise. */
typedef struct ekp_coco_gt {
    const int *count;          /* [n_img]                  ground-truth people per image */
    const double *keypoints;   /* [n_img, max_gt, 17, 3]   (x, y, v) in COCO keypoint order */
    const double *bbox;        /* [n_img, max_gt, 4]       (x, y, w, h) */
    const double *area;        /* [n_img, max_gt] */
    const int *iscrowd;        /* [n_img, max_gt] */
    const int *ignore;         /* [n_img, max_gt]          iscrowd || num_keypoints == 0 */
} ekp_coco_gt;
typedef struct ekp_coco_dt {
    const int *count;          /* [n_img]                  detections per image */
    const double *keypoints;   /* [n_img, max_dt, 17, 3] */
    const double *score;       /* [n_img, max_dt] */
} ekp_coco_dt;
typedef struct ekp_coco_eval_out {
    double *precision;         /* [T, R, A]   accumulate()'s precision[:, :, 0, :, 0] */
    double *recall;            /* [T, A]      recall[:, 0, :, 0] */
    double *scores;            /* [T, R, A]   scores[:, :, 0, :, 0] */
    /* optional (NULL: not written), for tests; dt index d = the rank in the image's score order */
    int *dt_match;             /* [n_img, A, T, max_det]   the matched gt row, or -1 (also for d past the kept dts) */
    int *dt_ignore;            /* [n_img, A, T, max_det]   evaluateImg's dtIgnore (0 past the kept dts) */
    double *oks;               /* [n_img, max_det, max_gt] computeOks' matrix, gts in row order (0 past the counts) */
} ekp_coco_eval_out;
/* Limits.  The per-image OKS matrix (max_det x max_gt float64) lives in the shared memory of the image's block, beside
 * the image's sort keys (max_dt) and one matched flag per walk and gt: at the limits 116.7 of the 227 KB a block has. */
#define EKP_COCO_LIMIT_CURVES 32       /* T * A: one tp and one fp bit per curve and detection */
#define EKP_COCO_LIMIT_REC 1024        /* R */
#define EKP_COCO_LIMIT_GT 128          /* max_gt */
#define EKP_COCO_LIMIT_DT 1024         /* max_dt */
#define EKP_COCO_LIMIT_DET 100         /* max_det */
#define EKP_COCO_LIMIT_IMAGES 1048576  /* n_img */
/* Bytes of the workspace of one evaluation (256-byte aligned); 0 when a size is outside its limit.  It grows with
 * n_img x max_det (about 51 bytes a slot), and does not depend on max_gt, max_dt or n_iou. */
long long ekp_coco_eval_workspace_bytes(int n_img, int max_gt, int max_dt, int max_det, int n_area, int n_iou);
/* One evaluation, asynchronous on `stream`: 29 kernel launches (one block per image, eight 8-bit passes of a radix sort
 * of n_img x max_det slots, four accumulate steps), counted in ekp_kernel_launches; no host wait, no allocation.  Every
 * output entry is written.  The workspace is the caller's (at least ekp_coco_eval_workspace_bytes), may be reused by
 * calls ordered after this one, must be 256-byte aligned, and is not read before it is written.  The context supplies the device, the error
 * reporting and the launch count.  EKP_ERR_ARG for a NULL context, table or required output, a size outside its limit
 * (n_img, max_gt, max_dt, max_det, T, R, A >= 1; T * A <= EKP_COCO_LIMIT_CURVES) or a pointer that is not 8-byte
 * aligned. */
int ekp_coco_eval_kpts(ekp_ctx *ctx, const ekp_coco_gt *gt, int max_gt, const ekp_coco_dt *dt, int max_dt, int n_img,
                       int max_det, const double *iou_thrs, int T, const double *rec_thrs, int R, const double *area_rng,
                       int A, void *workspace, const ekp_coco_eval_out *out, void *stream);
/* Test hook for ekp_coco_eval_kpts: the same per-image and accumulate code run serially on the CPU on HOST buffers (the
 * radix sort replaced by std::stable_sort on the same keys), with the same checks.  It is not a CPU path. */
int ekp_debug_coco_eval_host(const ekp_coco_gt *gt, int max_gt, const ekp_coco_dt *dt, int max_dt, int n_img, int max_det,
                             const double *iou_thrs, int T, const double *rec_thrs, int R, const double *area_rng, int A,
                             const ekp_coco_eval_out *out);

/* ---- drawing (SURVEY.md 8f row f2) --------------------------------------------------------------
 * Paints the people of the last run onto n DEVICE frames uint8 [n, H, W, 3] (contiguous, in place), as the reference's
 * draw_humans (lib/utils/common.py:252-275) paints each image's list[Human]: byte for byte.  Per human of the table, in
 * table order, its part markers (cv2.circle radius 3, thickness 3) in part order, then its limbs (cv2.line thickness 3)
 * in CocoPairsRender order; a pixel takes the colour of the last of them that covers it, CocoColors written to channels
 * 0, 1, 2 in tuple order.  Coordinates are normalised by the last run's full-resolution map (8h x 8w; H x W of
 * ekp_process_paf_dev's paf_mat), so frames of any size up to EKP_DRAW_MAX_SIDE a side work.  Pixels no marker or limb
 * covers are not touched.  Asynchronous on `stream`, ordered after the run; no host wait.  Draws what the human table
 * holds, overflow or not (ekp_results* report overflow).  Two kernel launches (counted in ekp_kernel_launches); a
 * context-owned key buffer of n x H x W uint32 is allocated on first use and grown on demand.  The draw is ordered
 * before the context's next run on any stream, so a run cannot overwrite the results the draw reads.
 * EKP_ERR_STATE before any run; EKP_ERR_ARG for a NULL context or frames, n != ekp_last_batch(ctx), or H, W outside
 * [1, EKP_DRAW_MAX_SIDE]. */
#define EKP_DRAW_MAX_SIDE 16384
int ekp_draw_humans(ekp_ctx *ctx, unsigned char *frames, int n, int H, int W, void *stream);

/* Test hooks for the rasteriser of ekp_draw_humans: the same code, run serially on the CPU on HOST buffers (they are not a
 * CPU path of ekp_draw_humans).  ekp_debug_raster_host sets mask[y][x] = 1 (uint8 [H, W]) for every pixel one primitive
 * paints: kind 1 the part marker centred at (x0, y0), kind 2 the limb (x0, y0) - (x1, y1).  ekp_debug_draw_host paints
 * the people of a human table (num_humans [n], parts ekp_peak [n, max_humans, 18] as ekp_results_humans writes it)
 * normalised by a map_h x map_w map onto frames uint8 [n, H, W, 3], in drawing order. */
int ekp_debug_raster_host(int kind, int x0, int y0, int x1, int y1, int H, int W, unsigned char *mask);
int ekp_debug_draw_host(const int *num_humans, const ekp_peak *parts, int max_humans, int map_h, int map_w,
                        unsigned char *frames, int n, int H, int W);

/* The 13 distinct weights w[-12] .. w[0] of scipy.ndimage's Gaussian kernel for sigma = 3 as the context uploads them for
 * EKP_FRONTEND_REFERENCE_GAUSS (host-only; tests compare them with scipy's own array). */
int ekp_scipy_gauss3_weights(double *out13);

/* Test hook: sorts scores (descending, comparator `a.score > b.score`, pafprocess.cpp:244-246) and
 * the tags riding along with the device code's replay of libstdc++'s std::sort, in place, DEVICE
 * pointers.  The resulting permutation of equal scores must equal the reference's (tests). */
int ekp_debug_std_sort(ekp_ctx *ctx, float *scores, unsigned *tags, int n, void *stream);

/* Per-part offsets into the peak table of the last run: int [n, 19]; part k of image i occupies
 * rows part_off[i][k] .. part_off[i][k+1]-1 of peaks_line (part_off[i][18] == n_peaks[i]). */
int ekp_results_parts(ekp_ctx *ctx, int *part_off);

/* Debug / test access to the dense front-end's smoothed map: float32 [n, 8h, 8w, 18] DEVICE. */
int ekp_dense_smooth_debug(ekp_ctx *ctx, const float *heat, int n, int h, int w, int layout, float *smooth_out,
                           void *stream);

/* ---- input side (SURVEY.md 8f row f4) --------------------------------------------------------
 * Geometry of the reference's `padding` (lib/evaluate/estimator.py:52-68): the long side is scaled
 * to dest_size (cv2.resize, INTER_LINEAR), then zero-padded to a multiple of `factor`. */
int ekp_preprocess_dims(int src_h, int src_w, int dest_size, int factor, int *resized_h, int *resized_w,
                        int *padded_h, int *padded_w, double *scale);
/* padding + vgg_preprocess (mode 0) / rtpose_preprocess (mode 1) (lib/datasets/preprocessing.py:16-43)
 * for n equally sized uint8 BGR frames [n, src_h, src_w, 3] (DEVICE) -> float32 [n, 3, padded_h,
 * padded_w] (DEVICE), bit-identical to the reference's Python. */
int ekp_preprocess(ekp_ctx *ctx, const unsigned char *frames, int n, int src_h, int src_w, int dest_size,
                   int factor, int mode, float *out, void *stream);

/* Per-stage device timing for the benchmark.  When enabled, CUDA events are recorded on the work
 * stream around each stage of every run (a ring of the last 64 runs).  ekp_stage_times waits for
 * the stream and returns the mean milliseconds of: [0] stages 1-3 (front-end kernel(s); for 16-bit inputs
 * also the widening kernel of the *_typed entry points),
 * [1] peak sort, [2] stage 4 + sort/greedy (paf_connect), [3] assembly; *runs = runs averaged. */
int ekp_set_timing(ekp_ctx *ctx, int enable);
int ekp_stage_times(ekp_ctx *ctx, float *ms, int *runs);

/* Introspection for tests and the benchmark. */
int ekp_last_batch(const ekp_ctx *ctx);   /* images of the last submitted run = rows the ekp_results* calls write */
int ekp_max_batch(const ekp_ctx *ctx);
int ekp_max_peaks(const ekp_ctx *ctx);
int ekp_max_humans(const ekp_ctx *ctx);
int ekp_max_part(const ekp_ctx *ctx);
int ekp_max_cand(const ekp_ctx *ctx);
long long ekp_kernel_launches(const ekp_ctx *ctx); /* kernels launched by this context so far */
long long ekp_graph_launches(const ekp_ctx *ctx);  /* batches of those that were replayed as a CUDA graph */

/* Pinned (page-locked) host memory for ekp_postprocess_host: when a batch's heat tensor is directly followed by its
 * PAF tensor in ONE such block the library moves both with a single copy.  write_combined != 0 asks for
 * write-combined memory (CPU writes only, sequential). */
int ekp_host_alloc(void **out, size_t bytes, int write_combined);
/* Releasing a block also retires the CUDA graphs of host-entry batches captured before it (they are captured again on
 * their next submission), so a new block that comes back at the address of a released one is never read through a
 * graph of the old one. */
int ekp_host_free(void *p);

/* ---- the reference operator surface (lib/pafprocess/pafprocess.h:53-59) ------------------
 * HOST pointers.  peaks [p1,p2,p3] rows (x, y, score, _, part); heatmap [h1,h2,h3] is used only
 * through h1 and is never read (as in the reference, pafprocess.cpp:83) so it may be NULL;
 * pafmap [f1,f2,f3].  Runs on the device selected by EKP_DEVICE (default 0).  Unlike the
 * reference (always 0, undefined behaviour on bad input) a negative ekp_status is returned
 * when the input is invalid or no GPU is available.
 * Only what stage 4 reads of pafmap crosses the bus: the <= 10 sample positions of every candidate pair are listed
 * (on the host for up to 64 Ki samples: one upload, one download, no wait in between; by a kernel beyond that), the two
 * floats at each position are gathered from the caller's array and uploaded.  Environment EKP_PROCESS_PAF_UPLOAD =
 * listed (default) | sparse (always list on the device) | dense (upload the whole tensor). */
int process_paf(int p1, int p2, int p3, float *peaks, int h1, int h2, int h3, float *heatmap, int f1, int f2,
                int f3, float *pafmap);
int get_num_humans(void);
int get_part_cid(int human_id, int part_id);
float get_score(int human_id);
int get_part_x(int cid);
int get_part_y(int cid);
float get_part_score(int cid);

#ifdef __cplusplus
}
#endif
#endif /* EKPOSE_B200_H */
