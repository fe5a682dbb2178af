/*
 * ofb200.h -- C ABI of the B200-native dense pyramidal Lucas-Kanade path.
 *
 * Drop-in boundary for ONE path of Kr-Stam/CUDA_Optical_Flow_2: Gaussian pyramid -> Ix/Iy/It ->
 * windowed structure-tensor sums -> per-pixel 2x2 solve -> coarse-to-fine flow upsample + warp.
 * Every entry point names the reference interface it replaces (file:line into the reference tree).
 * Plain pointers and sizes only; no C++ or torch types.  All functions return OFB_OK (0) or an
 * OFB_ERR_* code; ofb_last_error() gives the message of the calling thread's last failure.
 * There is no CPU fallback: without a CUDA device every compute entry point fails with OFB_ERR_CUDA.
 *
 * Layouts
 *   host images (reference layout): u8, 3 interleaved channels, tightly packed, channels equal
 *       (OptFlowGpu.cu:58-59); the LK stages read channel 0 only (OptFlowGpu.cu:1081).
 *   device images (hot path):       u8, planar, row pitch a multiple of 16 bytes, base 16-byte
 *       aligned; image i of a batch starts at base + i*image_stride_bytes (multiple of 16).
 *   flow: float (u,v) interleaved per pixel, tightly packed rows (OptFlowGpu.cu:1844-1845);
 *       level k of a pyramid is (w>>k) x (h>>k) pixels (main.cu:95-104).
 */
#ifndef OFB200_H
#define OFB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OFB_OK 0
#define OFB_ERR_INVALID 1     /* bad argument */
#define OFB_ERR_CUDA 2        /* CUDA runtime / driver failure (including "no device") */
#define OFB_ERR_UNSUPPORTED 3 /* valid request outside the built configuration set */
#define OFB_ERR_NOMEM 4

/* How next_k is shifted back by the coarser flow before a level is solved
 * (cpu::shift_back_pyramid, OptFlowCPU.cpp:241-282, called at OptFlowGpu.cu:1918-1922). */
#define OFB_WARP_AS_WRITTEN 0 /* bug-compatible: the flow of pixel (0,0) of every coarser level, nearest */
#define OFB_WARP_NEAREST 1    /* per-pixel coarser flow (index i>>off as main.cu:141-143), nearest sample */
#define OFB_WARP_BILINEAR 2   /* per-pixel coarser flow, 8.8 fixed-point bilinear sample (north_star) */

/* The per-pixel 2x2 solve of the fused level kernel (g_inv_matrix_float, OptFlowGpu.cu:1819-1846).  Both modes solve
 * the same system from the same exact integer window sums; non-finite outputs (det == 0) fall on the same pixels.
 *   EXACT (default): the reference's double-precision operation order; flow bit-identical to the reference's solve.
 *   FAST           : exact 64-bit integer determinant and numerators, each rounded once to float, one hardware
 *                    reciprocal: |du|, |dv| <= 1e-4 px + 1e-5 |ref| per level on identical inputs (measured: a few
 *                    float ulps, < 3e-7 relative); about 20 % less time in the level kernel.  Pixels whose |SIxIy|
 *                    exceeds 94,906,265 (b*b no longer exact in double: the reference's determinant of a
 *                    one-dimensional window is then a rounding residue, not 0) take the EXACT sequence and match it
 *                    bit for bit; windows up to 9 never reach that. */
#define OFB_SOLVE_EXACT 0
#define OFB_SOLVE_FAST 1

#define OFB_MAX_LEVELS 8
#define OFB_MAX_WINDOW 19 /* odd windows 3..19; 19 is what OptFlowGpu.cu:1944-1945 hard-codes */

typedef struct ofb_ctx ofb_ctx; /* owns device workspace, streams and TMA descriptors for one GPU */

/* Parameters of one pyramidal solve (the hard-coded values of main.cu:192 and OptFlowGpu.cu:1944). */
typedef struct ofb_params {
    int w, h;         /* level-0 width / height in pixels */
    int levels;       /* pyramid levels, 1..OFB_MAX_LEVELS (main.cu:192 uses 4) */
    int win;          /* LK window, odd, 3..OFB_MAX_WINDOW */
    int warp_mode;    /* OFB_WARP_* */
    float flow_scale; /* multiplies the coarser flow before the warp; 1.0f = the reference (Q5) */
    int n_pairs;      /* frame pairs in the batch (>= 1) */
} ofb_params;

const char *ofb_last_error(void);
int ofb_version(void);

/* One context per GPU (and per host thread that drives it).  Replaces the reference's implicit
 * device 0 + per-call cudaMalloc/cudaFree (OptFlowGpu.cu:1105-1106, 1123-1124). */
int ofb_ctx_create(int device, ofb_ctx **out);
int ofb_ctx_destroy(ofb_ctx *ctx);
int ofb_ctx_device(const ofb_ctx *ctx, int *device);
int ofb_ctx_sm_count(const ofb_ctx *ctx, int *sm_count);
/* Threads and streams.  A context belongs to one host thread at a time.  All entry points share the context's one
 * device workspace: a call on a stream waits (on the device, cudaStreamWaitEvent) for the previous call's use of it on
 * another stream, so results are correct whatever streams are mixed, but two streams of one context never overlap --
 * use one context per stream for that.  The workspace grows on demand; growing synchronises the device and frees the
 * old block, which invalidates CUDA graphs captured from earlier calls: size it first with ofb_ctx_reserve_pairs.  A call made
 * while its stream is being captured takes no part in that ordering (replays are ordered by their caller). */
int ofb_ctx_reserve_pairs(ofb_ctx *ctx, const ofb_params *p); /* workspace for ofb_flow_pairs_device with these parameters */
/* Solve mode (OFB_SOLVE_*) of every fused-LK launch made through this context from now on. */
int ofb_ctx_set_solve(ofb_ctx *ctx, int solve_mode);
int ofb_ctx_get_solve(const ofb_ctx *ctx, int *solve_mode);
/* Host threads of the batched host entry points (ofb_flow_pairs_host / _ex) for 3-channel input, 0..64, default 0 (or
 * OFB_HOST_THREADS in the environment).  The reference's host images are 3-channel and its kernels read channel 0
 * (OptFlowGpu.cu:1040-1090).  With 0 all three channels are uploaded and the device drops two; with n > 0 a pool of n
 * host threads (the caller's included) extracts channel 0 into pinned staging buffers while earlier sub-batches are in
 * flight and a third of the bytes cross PCIe -- the results are identical.  The end-to-end path is bound by PCIe bytes,
 * so this is what bench.py's `e2e` record runs with. */
int ofb_ctx_set_host_threads(ofb_ctx *ctx, int threads);
int ofb_ctx_get_host_threads(const ofb_ctx *ctx, int *threads);
/* The extraction itself (host only, no device involved): dst_planar[i] = src_c3[3 * i], i < n_pixels, on `threads`
 * host threads (1..64). */
int ofb_c3_extract_host(const unsigned char *src_c3, unsigned char *dst_planar, size_t n_pixels, int threads);

/* ------------------------------------------------------------------------------------------
 * Device-resident hot path (what the metric is quoted on).  Asynchronous on `stream`
 * (a cudaStream_t passed as void*; NULL = the legacy default stream).
 * ---------------------------------------------------------------------------------------- */

/* Whole path for a batch of pairs: pyramids of both frames (gpu::gauss_pyramid,
 * OptFlowGpu.cu:1262-1271) then the coarse-to-fine loop of main.cu:256-262 calling the fused
 * per-level kernel (gpu::calc_opt_flow, OptFlowGpu.cu:1909-1979).
 *   prev_d / next_d : level-0 planar u8 frames, n_pairs images each.
 *   flow_levels_d[k]: out, RESIDUAL flow of level k (what the reference leaves in
 *                     optFlowPyramid[k]); n_pairs * (h>>k) * (w>>k) * 2 floats.
 *   total_flow_d    : optional out (may be NULL), the composition rule of main.cu:136-147 at
 *                     level 0: sum_k 2^k * flow_k[i>>k, j>>k]; n_pairs * h * w * 2 floats.
 * At most 65535 pairs per call (as ofb_lk_level_device and ofb_flow_pairs_fb_device). */
int ofb_flow_pairs_device(ofb_ctx *ctx, const ofb_params *p, const uint8_t *prev_d, const uint8_t *next_d,
                          size_t pitch_bytes, size_t image_stride_bytes, float *const *flow_levels_d,
                          float *total_flow_d, void *stream);

/* One pyramid step for n_images planar images: dst = (sw>>1) x (sh>>1).
 * Replaces gpu::gauss_pyramid_level / g_gauss_pyramid (OptFlowGpu.cu:1235-1259, 1198-1232). */
int ofb_pyr_down_device(ofb_ctx *ctx, const uint8_t *src_d, size_t src_pitch, size_t src_image_stride, int sw, int sh,
                        uint8_t *dst_d, size_t dst_pitch, size_t dst_image_stride, int n_images, void *stream);

/* Two pyramid steps in one launch: dst1 = (sw>>1) x (sh>>1) and dst2 = (sw>>2) x (sh>>2), byte-identical to two
 * ofb_pyr_down_device calls (gpu::gauss_pyramid's loop over levels, OptFlowGpu.cu:1262-1290), but level +1 is not read
 * back from memory: the kernel forms level +2 from the bytes it has just produced.  What the batch entry points use
 * while at least two levels are left to build. */
int ofb_pyr_down2_device(ofb_ctx *ctx, const uint8_t *src_d, size_t src_pitch, size_t src_image_stride, int sw, int sh,
                         uint8_t *dst1_d, size_t dst1_pitch, size_t dst1_image_stride, uint8_t *dst2_d, size_t dst2_pitch,
                         size_t dst2_image_stride, int n_images, void *stream);

/* Row-strip variant of ofb_pyr_down_device for frames partitioned across GPUs: the source buffer
 * holds global rows [src_y_off, src_y_off + src_rows) of a level of width sw; destination rows
 * [dst_y0, dst_y1) (global numbering) of the next level are written to dst_d, whose row 0 is
 * global row dst_y0.  Source rows 2y-1 .. 2y+1 must be present for every destination row y. */
int ofb_pyr_down_strip_device(ofb_ctx *ctx, const uint8_t *src_d, size_t src_pitch, int sw, int src_rows,
                              int src_y_off, uint8_t *dst_d, size_t dst_pitch, int dst_y0, int dst_y1, void *stream);

/* One fused LK level on device-resident planar images: warp next by the coarser cumulative flow,
 * Ix/Iy/It, five window sums, solve.  Replaces the body of gpu::calc_opt_flow for one level
 * (OptFlowGpu.cu:1909-1979) without its host round trips.
 *   cum_in_d : cumulative flow of the next-coarser level ((w>>1) x (h>>1) float2 per pair:
 *              cum_{k+1} = flow_{k+1} + 2*cum_{k+2}[i>>1, j>>1]); NULL for the coarsest level
 *              (not warped, OptFlowGpu.cu:1918).
 *   flow_out_d: residual flow of this level.  cum_out_d: optional, 2*cum_in[i>>1,j>>1] + flow.
 *   n_pairs: at most 65535. */
int ofb_lk_level_device(ofb_ctx *ctx, const uint8_t *prev_d, const uint8_t *next_d, size_t pitch_bytes,
                        size_t image_stride_bytes, int w, int h, int n_pairs, int win, int warp_mode, float flow_scale,
                        const float *cum_in_d, float *flow_out_d, float *cum_out_d, void *stream);

/* Row-strip variant of ofb_lk_level_device for frames partitioned across GPUs.  The buffers hold
 * rows [y_off, y_off + h_local) of a (w x h_global) level; flow is produced for local rows
 * [out_y0, out_y1).  cum_in_d holds coarse rows starting at global coarse row cum_y_off
 * (cum_h_local rows).  Rows of prev/next needed beyond the local buffer must be halo rows already
 * exchanged by the caller; only the global image border is zero padded. */
int ofb_lk_level_strip_device(ofb_ctx *ctx, const uint8_t *prev_d, const uint8_t *next_d, size_t pitch_bytes, int w,
                              int h_local, int y_off, int h_global, int out_y0, int out_y1, int win, int warp_mode,
                              float flow_scale, const float *cum_in_d, int cum_y_off, int cum_h_local,
                              float *flow_out_d, float *cum_out_d, int *reach_overflow_d, void *stream);

/* Layout helpers: channel 0 of 3-channel interleaved u8 -> planar pitched u8 and back
 * (the reference keeps 3 equal channels; grayscale_avg OptFlowGpu.cu:58-59). */
int ofb_c3_to_planar_device(ofb_ctx *ctx, const uint8_t *src_c3_d, int w, int h, int n_images, uint8_t *dst_d,
                            size_t dst_pitch, size_t dst_image_stride, void *stream);

/* ------------------------------------------------------------------------------------------
 * Host-pointer entry points with the reference's argument meaning (synchronous, like the
 * reference's blocking cudaMemcpy).  These are what the C++ `namespace gpu` wrappers in
 * include/OptFlowGpuB200.hpp forward to.
 * ---------------------------------------------------------------------------------------- */

/* gpu::gauss_pyramid(unsigned char** pyramid, int w, int h, int levels, mask, mw, mh),
 * OptFlowGpu.cuh:21 / OptFlowGpu.cu:1262.  3-channel interleaved host levels, pyramid[0] is the
 * input; the reference ignores its mask arguments (fixed 3x3 binomial), so they are not taken. */
int ofb_gauss_pyramid_host_u8c3(ofb_ctx *ctx, unsigned char **pyramid, int w, int h, int levels);

/* gpu::calc_opt_flow(prev, next, w, h, optFlowPyramid, level, maxLevel), OptFlowGpu.cuh:33 /
 * OptFlowGpu.cu:1909, with the window (hard-coded 19 there), warp mode and flow scale exposed.
 * prev/next are level `level` images (3-ch interleaved host); optFlowPyramid[k > level] are read,
 * optFlowPyramid[level] is written; w,h are this level's size. */
int ofb_calc_opt_flow_host_u8c3(ofb_ctx *ctx, const unsigned char *prev, const unsigned char *next, int w, int h,
                                float **optFlowPyramid, int level, int maxLevel, int win, int warp_mode,
                                float flow_scale);

/* gpu::conv_3ch_1ch_tiled_uchar_float(src_h, w, h, dest_h, mask_t, mw, mh), OptFlowGpu.cuh:17 /
 * OptFlowGpu.cu:1100: correlation of channel 0 with an mw x mh (<= 5x5) mask, zero padding. */
int ofb_conv_3ch_1ch_u8_f32_host(ofb_ctx *ctx, const unsigned char *src_h, int w, int h, float *dest_h,
                                 const float *mask, int mw, int mh);

/* gpu::srm_1ch_float(arr1_h, arr2_h, w, h, ww, wh, dest_h), OptFlowGpu.cuh:25 / OptFlowGpu.cu:1597:
 * windowed sum of products, fp32 running sum in the reference's tap order. */
int ofb_srm_1ch_f32_host(ofb_ctx *ctx, const float *arr1_h, const float *arr2_h, int w, int h, int ww, int wh,
                         float *dest_h);

/* gpu::inverse_matrix_float(sumIx2, sumIy2, sumIxIy, sumIxIt, sumIyIt, optFlowPyramid, level, w, h),
 * OptFlowGpu.cuh:31 / OptFlowGpu.cu:1858: per-pixel 2x2 solve in double, writes optFlowPyramid[level]. */
int ofb_inverse_matrix_f32_host(ofb_ctx *ctx, const float *sumIx2, const float *sumIy2, const float *sumIxIy,
                                const float *sumIxIt, const float *sumIyIt, float **optFlowPyramid, int level, int w,
                                int h);

/* The loop of main.cu:246-262 for a batch of pairs with HOST buffers: upload level-0 frames
 * (channels = 3: reference layout, channel 0 is used; channels = 1: planar gray), build both
 * pyramids, run all levels, download the residual flow of every level.
 *   flow_levels_h[k]: n_pairs * (h>>k) * (w>>k) * 2 floats.  Pinned host memory makes the copies
 * asynchronous; pageable memory works too. */
int ofb_flow_pairs_host(ofb_ctx *ctx, const ofb_params *p, const unsigned char *prev_h, const unsigned char *next_h,
                        int channels, float *const *flow_levels_h);
/* The same loop with the outputs chosen by the caller: flow_levels_h may be NULL or hold NULL entries (levels that stay
 * on the device), total_flow_h (may be NULL) receives the level-0 composition of main.cu:136-147, n_pairs * h * w * 2
 * floats -- what visualizeFlowField consumes.  Planar gray in (channels = 1) and the total flow only out moves 10 bytes
 * per pixel over PCIe instead of the 16.5 of the reference layout with every level. */
int ofb_flow_pairs_host_ex(ofb_ctx *ctx, const ofb_params *p, const unsigned char *prev_h, const unsigned char *next_h,
                           int channels, float *const *flow_levels_h, float *total_flow_h);

/* ------------------------------------------------------------------------------------------
 * Pre-processing and the frame loop of main.cu (SURVEY.md 8f rows 1-3)
 * ---------------------------------------------------------------------------------------- */

/* gpu::grayscale_avg(src_h, dest_h, h, w), OptFlowGpu.cuh:5 / OptFlowGpu.cu:47-95: (c0+c1+c2)/3 into all
 * three channels.  NOTE the reference's argument order: height before width. */
int ofb_grayscale_avg_host_u8c3(ofb_ctx *ctx, const unsigned char *src_h, unsigned char *dest_h, int h, int w);

/* gpu::bilinear_filter(src, gray, dest, w, h, ww, wh, sigmaS, sigmaB), OptFlowGpu.cuh:35 /
 * OptFlowGpu.cu:1984-2083: despite the name a bilateral filter (spatial Gaussian sigmaS x range Gaussian
 * sigmaB on gray channel 0), double precision, square odd window up to 9x9, 3-channel host images. */
int ofb_bilinear_filter_host_u8c3(ofb_ctx *ctx, const unsigned char *src, const unsigned char *gray, unsigned char *dest,
                                  int w, int h, int ww, int wh, double sigmaS, double sigmaB);

/* The same filter on a device-resident planar gray image (src == gray, the way main.cu:240 uses it). */
int ofb_bilateral_planar_device(ofb_ctx *ctx, const uint8_t *gray_d, size_t pitch, int w, int h, int ww, int wh,
                                double sigmaS, double sigmaB, uint8_t *dst_d, size_t dst_pitch, void *stream);

/* Frame sequence in the role of main.cu:222-275.  Each pushed BGR frame (3-channel interleaved host
 * buffer) is uploaded once, converted to gray (main.cu:232), optionally bilateral-filtered (main.cu:240;
 * bil_win = 0 disables it), turned into a pyramid (main.cu:250) and solved against the PREVIOUS frame's
 * pyramid, which stays on the device (the swap of main.cu:270-272) -- half the pyramid work and no
 * re-upload.  The first push only primes the pyramid (*has_flow = 0).
 *   flow_levels_h[k]: residual flow of level k, (h>>k)*(w>>k)*2 floats; total_flow_h: optional level-0
 *   composition (main.cu:136-147). */
typedef struct ofb_stream ofb_stream;
int ofb_stream_create(ofb_ctx *ctx, const ofb_params *p, int bil_win, double bil_sigma_s, double bil_sigma_b,
                      ofb_stream **out);
int ofb_stream_push_bgr_host(ofb_stream *s, const unsigned char *frame_bgr, float *const *flow_levels_h,
                             float *total_flow_h, int *has_flow);
int ofb_stream_destroy(ofb_stream *s);

/* ---- row strips of one large pair over several GPUs (BASELINE configs[4]); the reference is single-GPU ----------
 * One process per GPU, one handle per process.  The schedule (strip bounds fixed on the coarsest level and doubled
 * per finer level; per level the neighbours' image halo rows and the next-coarser cumulative-flow rows) is that of
 * cuda_optical_flow_2_b200/dist.py; here a whole pair is enqueued on one stream without host synchronisation.
 * The result is bit-identical to the whole-frame result unless ofb_strips_check reports that a warp sample reached
 * past the exchanged rows (`reach`, in rows of the level being warped).
 * The halo rows move through peer memory.  After ofb_strips_create (not a collective) every rank of a world > 1
 * publishes ofb_strips_peer_handle (128 bytes: a CUDA IPC handle of the one allocation its neighbours write into), the
 * application all-gathers the blobs and hands them to ofb_strips_peer_connect.  An exchange is then a store of the
 * sender's kernels into the receiver's memory over NVLink plus an epoch flag raised there, and a wait for that flag on the
 * receiver's stream.  ofb_strips_peer_connect_local does the same for ranks living in one process.
 *   ofb_strips_plan_query     : host only, no device: the rows {y0, y1, by0, by1, cy0, cy1, eb0, eb1} of a level on a rank
 *   plans refused (ofb_strips_plan_query, _create, _create_fb alike, on every rank): OFB_ERR_INVALID when the coarsest
 *                               level has fewer rows than ranks (or no column); OFB_ERR_UNSUPPORTED when strips are so
 *                               much thinner than their halo that, on ANY rank, one exchange of a pair would send rows to
 *                               or receive rows from more than 4 ranks, the image exchange would copy more than 8 row
 *                               segments, or more than 8 ranks would push to, or be pushed to by, one rank over a pair
 *                               (_create_fb: with its check-row and backward exchanges).  ofb_last_error names the
 *                               exchange, the rank and the count; fewer ranks, fewer levels or a smaller reach / fb_reach
 *                               help.  Plans whose coarsest strips are 1 or 2 rows are refused on more than 5 ranks
 *   ofb_strips_check        : synchronises; *overflow bit 0 = a warp sample reached past the halo rows, bit 1 = a
 *                               neighbour's rows did not arrive within 4 s, bit 2 = a checked pair's check needed a
 *                               backward tap outside the rows the rank holds (OFB_FB_UNCHECKED pixels: raise fb_reach).
 *                               The flag is sticky: it covers every pair since the previous check, which clears it
 *   ofb_strips_run_phase_device: one of the 2 * levels phases of a pair: 0 = upload + push of the level-0 image rows;
 *                               1 = wait, pyramid, coarsest level; 2j = push of the cumulative flow of level L-j;
 *                               2j+1 = wait, level L-1-j (j = 1 .. L-1).  A host that runs several ranks in ONE process
 *                               on ONE stream (tests on a single GPU) enqueues phase p of every rank before phase p+1 of
 *                               any: no kernel then ever waits for a kernel enqueued after it
 *   ofb_strips_destroy        : waits (bounded) until every neighbour has acknowledged this rank's last pair before its
 *                               arena is unmapped and freed; all ranks must have run the same number of pairs.  Across
 *                               processes also put a barrier between the last check and the destroy calls
 *   ofb_strips_run_device     : prev_own_d / next_own_d = rows [y0, y1) of level 0 (ofb_strips_own_rows), planar u8
 *   ofb_strips_result         : device pointers to the own rows of the residual flow / cumulative flow of a level
 *   ofb_strips_input          : where the own rows of level 0 live inside the handle: a producer that writes them there
 *                               and passes the same pointers to ofb_strips_run_device saves the upload copy
 *   ofb_strips_set_total      : whether level 0 also writes the total flow of the pair (default on) */
typedef struct ofb_strips ofb_strips;
int ofb_strips_plan_query(int w, int h, int levels, int win, int world, int rank, int reach, int level, int *out8);
int ofb_strips_create(ofb_ctx *ctx, int w, int h, int levels, int win, int warp_mode, float flow_scale, int world, int rank,
                      int reach, ofb_strips **out);
int ofb_strips_own_rows(const ofb_strips *s, int level, int *y0, int *y1);
int ofb_strips_run_device(ofb_strips *s, const uint8_t *prev_own_d, const uint8_t *next_own_d, size_t pitch, void *stream);
int ofb_strips_run_phase_device(ofb_strips *s, const uint8_t *prev_own_d, const uint8_t *next_own_d, size_t pitch, int phase,
                                void *stream);
int ofb_strips_result(const ofb_strips *s, int level, float **flow_own_d, float **total_own_d);
int ofb_strips_check(ofb_strips *s, void *stream, int *overflow);
int ofb_strips_destroy(ofb_strips *s);
int ofb_strips_input(const ofb_strips *s, uint8_t **prev_own_d, uint8_t **next_own_d, size_t *pitch);
int ofb_strips_set_total(ofb_strips *s, int on);
int ofb_strips_set_fused(ofb_strips *s, int on); /* peer memory: halo rows pushed by the level kernels themselves (default on) */
int ofb_strips_peer_handle(ofb_strips *s, void *blob128);
int ofb_strips_peer_connect(ofb_strips *s, const void *blobs_world_x_128);
int ofb_strips_peer_arena(ofb_strips *s, void **arena_d);
int ofb_strips_peer_connect_local(ofb_strips *s, void *const *arenas_d);

/* ---- forward-backward consistency check on row strips (a checked pair) --------------------------------------------
 * The check of ofb_flow_pairs_fb_device on one pair cut into row strips.  A checked pair runs the forward level loop as
 * ofb_strips_run_device does (level 0 always writes the total flow), then the backward level loop (next -> prev) on the
 * pyramid the rank has already built (no second image exchange), then exchanges the backward total rows the neighbours'
 * checks sample and checks the own rows [y0, y1) of level 0.  All of it is enqueued on one stream without host
 * synchronisation, so a checked pair can be captured as a CUDA graph.
 *   ofb_strips_create_fb : the arguments of ofb_strips_create plus fb_reach >= 0, the level-0 rows beyond its own rows a
 *                          rank's check may sample: it holds backward total rows [max(0, y0 - fb_reach), min(h, y1 +
 *                          fb_reach + 1)).  The arena also holds the backward direction's regions, so a handle that runs
 *                          checked pairs is created this way (before ofb_strips_peer_handle / _connect).  flow_scale > 0.
 *                          Plain pairs (ofb_strips_run_device) run on it unchanged, and plain and
 *                          checked pairs may alternate; all ranks must be created with the same fb_reach.  Refuses
 *                          the plans ofb_strips_create refuses, and those whose check-row exchange or handshake goes
 *                          past the same limits (see the plans refused above).
 *   ofb_strips_run_fb_device : one checked pair; alpha >= 0, beta >= 0 as in ofb_flow_pairs_fb_device; want_err2 = 0 leaves
 *                          the err2 buffer untouched.  Bad arguments are refused before anything is enqueued.
 *   ofb_strips_run_fb_phase_device : one of its 4L + 1 phases (L = levels; ranks of one process on one stream, as
 *                          ofb_strips_run_phase_device):
 *                            0 .. 2L-1   the forward phases of ofb_strips_run_phase_device, without the handshake
 *                            2L          backward coarsest level L-1
 *                            2L+2j-1     push of the backward cumulative flow of level L-j        (j = 1 .. L-1)
 *                            2L+2j       wait, backward level L-1-j                               (j = 1 .. L-1)
 *                            4L-1        push of the own backward total rows the neighbours' checks sample
 *                            4L          wait, the check, the end-of-pair handshake
 *   ofb_strips_fb_result : device pointers to the own rows [y0, y1) of level 0: forward total, backward total (2 floats
 *                          per pixel), status (1 byte) and err2 (1 float) per pixel.
 * Status: that of ofb_fb_check_device, except that a pixel whose whole-frame status would read backward taps
 * (CONSISTENT, INCONSISTENT, BWD_NONFINITE) and has a tap of non-zero weight outside the rows held is OFB_FB_UNCHECKED
 * (err2 NaN; bit 2 of ofb_strips_check).  FWD_NONFINITE and OUTSIDE read no tap and are never replaced.  Unless
 * ofb_strips_check reports bit 0 or bit 2, every output is bit-identical to rows [y0, y1) of ofb_flow_pairs_fb_device on
 * the whole frame with the same parameters and solve mode. */
int ofb_strips_create_fb(ofb_ctx *ctx, int w, int h, int levels, int win, int warp_mode, float flow_scale, int world, int rank,
                         int reach, int fb_reach, ofb_strips **out);
int ofb_strips_run_fb_device(ofb_strips *s, const uint8_t *prev_own_d, const uint8_t *next_own_d, size_t pitch, float alpha,
                             float beta, int want_err2, void *stream);
int ofb_strips_run_fb_phase_device(ofb_strips *s, const uint8_t *prev_own_d, const uint8_t *next_own_d, size_t pitch, float alpha,
                                   float beta, int want_err2, int phase, void *stream);
int ofb_strips_fb_result(const ofb_strips *s, float **fwd_total_own_d, float **bwd_total_own_d, uint8_t **status_own_d,
                         float **err2_own_d);

/* ---- debug derivative views: showTest (main.cu:19-92) without the windows ------------------------------------------
 * ofb_conv_3ch_1ch_u8_u8_host replaces gpu::conv_3ch_1ch_tiled (OptFlowGpu.cuh; OptFlowGpu.cu:741-766, kernel
 *   :380-423): 3-channel u8 in (channel 0 is read), u8 out; an int accumulator truncated after every tap, result
 *   cast to unsigned char.
 * ofb_debug_view_host_u8c3: one window of showTest for pyramid level `level` (images of size w x h, 3-channel):
 *   OFB_VIEW_X: Dx_3x3 on cur (main.cu:44-56), OFB_VIEW_Y: Dy_3x3 on cur (:76-88), OFB_VIEW_T: Dt_3x3_n on cur minus
 *   on prev with unsigned char wrap-around (:57-75); then utils::cleanup_outliers and utils::upscale_1ch by
 *   2^level.  out_h: (w << level) * (h << level) bytes, values 0 / 255.  prev_level_h may be NULL for X and Y. */
#define OFB_VIEW_X 0
#define OFB_VIEW_Y 1
#define OFB_VIEW_T 2
int ofb_conv_3ch_1ch_u8_u8_host(ofb_ctx *ctx, const unsigned char *src_h, int w, int h, unsigned char *dest_h,
                                const float *mask, int mw, int mh);
int ofb_debug_view_host_u8c3(ofb_ctx *ctx, const unsigned char *prev_level_h, const unsigned char *cur_level_h, int w, int h,
                             int level, int which, unsigned char *out_h);

/* ---- flow composition and export: the headless part of visualizeFlowField (main.cu:114-174) --------------------
 * flow_pyramid_h[k]: residual flow of level k, (h>>k)*(w>>k)*2 floats, as gpu::calc_opt_flow leaves it
 * (main.cu:95-104, 256-262); only levels level..levels-1 are read.
 *
 * ofb_compose_flow_host: total_h[(i*(w>>level)+j)*2 + {0,1}] = sum_{k=levels-1..level} 2^(k-level) *
 *   flow_k[(i>>(k-level))*(w>>k) + (j>>(k-level))]  (main.cu:136-147, coarse to fine in float, bit for bit).
 * ofb_flow_arrows_host: the arrows main.cu:125-171 would draw: grid step (w>>level)/arrow_res, total flow clamped
 *   to +-step, end point truncated to int, arrows with a negative end point dropped.  arrows_xyxy receives up to
 *   max_arrows quadruples (x0, y0, x1, y1) in level pixels; *n_arrows is the full count.
 * ofb_write_flo: Middlebury .flo file (tag 202021.25f, int32 w, int32 h, w*h interleaved (u,v) floats): the file
 *   form of what the reference only shows on screen. */
int ofb_compose_flow_host(ofb_ctx *ctx, float *const *flow_pyramid_h, int w, int h, int levels, int level, float *total_h);
int ofb_flow_arrows_host(ofb_ctx *ctx, float *const *flow_pyramid_h, int w, int h, int levels, int level, int arrow_res,
                         int *arrows_xyxy, int max_arrows, int *n_arrows);
int ofb_write_flo(const char *path, const float *flow_h, int w, int h);

/* ---- forward-backward consistency check; the reference has no counterpart -----------------------------------------
 * Which flow values can be trusted: flow prev->next (f) and next->prev (b) should cancel where a pixel is visible in
 * both frames.  Per pixel (i, j), with s = flow_scale (px per flow unit, the ofb_params value), in this order:
 *   f = fwd[i][j] not finite                                         -> OFB_FB_FWD_NONFINITE (e.g. a det == 0 window, Q3)
 *   du = s*f.u, dv = s*f.v; !(|du| < 32768 && |dv| < 32768)           -> OFB_FB_OUTSIDE
 *   X = j*256 + rint(du*256), Y = i*256 + rint(dv*256) (half to even, the bilinear warp's 1/256-px rounding);
 *   X or Y outside [0, (w-1)*256] / [0, (h-1)*256]                   -> OFB_FB_OUTSIDE (the target leaves the frame)
 *   b = bilinear sample of bwd at (X/256, Y/256); a tap with weight 0 is not read; a read tap not finite
 *                                                                    -> OFB_FB_BWD_NONFINITE
 *   err2 = |s*(f + b)|^2, mag2 = |s*f|^2 + |s*b|^2 (px^2); err2 finite and err2 <= alpha*mag2 + beta
 *                                                                    -> OFB_FB_CONSISTENT, else OFB_FB_INCONSISTENT
 * (Sundaram, Brox and Keutzer 2010; alpha = 0.01, beta = 0.5 px^2 are the usual values.)  Every multiply and add is
 * rounded separately, without fma: the result does not depend on the compiler.  err2 (optional) receives the value
 * above for CONSISTENT / INCONSISTENT pixels and NaN for the others.  Flow fields are (u, v) float pairs in the
 * library's layout, pairs back to back (n_pairs*h*w*2 floats, 8-byte aligned); status is n_pairs*h*w bytes; err2
 * n_pairs*h*w floats (4-byte aligned) or NULL.  At most 65535 pairs per call and 32768 x 32768 pixels. */
#define OFB_FB_CONSISTENT 0
#define OFB_FB_INCONSISTENT 1
#define OFB_FB_OUTSIDE 2
#define OFB_FB_FWD_NONFINITE 3
#define OFB_FB_BWD_NONFINITE 4
#define OFB_FB_UNCHECKED 5 /* row strips only (ofb_strips_run_fb_device): a tap the check needs lies outside the rows held */
/* The check alone, on any two total-flow fields (e.g. the caller's own).  flow_scale > 0, alpha >= 0, beta >= 0. */
int ofb_fb_check_device(ofb_ctx *ctx, const float *fwd_d, const float *bwd_d, int w, int h, int n_pairs, float flow_scale,
                        float alpha, float beta, uint8_t *status_d, float *err2_d, void *stream);
/* Both directions of every pair plus the check.  The pyramids of both frames are built once (one launch, as in
 * ofb_flow_pairs_device); the level loop runs prev->next, then next->prev on the same pyramids.  fwd_total_d /
 * bwd_total_d (required, n_pairs*h*w*2 floats) receive the level-0 compositions (main.cu:136-147), bit-identical to
 * ofb_flow_pairs_device(prev, next) / ofb_flow_pairs_device(next, prev) with total_flow_d.  The residual pyramids of
 * both directions live in the context workspace.  p->flow_scale is the check's s and must be > 0. */
int ofb_flow_pairs_fb_device(ofb_ctx *ctx, const ofb_params *p, const uint8_t *prev_d, const uint8_t *next_d,
                             size_t pitch_bytes, size_t image_stride_bytes, float alpha, float beta, float *fwd_total_d,
                             float *bwd_total_d, uint8_t *status_d, float *err2_d, void *stream);
int ofb_ctx_reserve_pairs_fb(ofb_ctx *ctx, const ofb_params *p); /* workspace for the call above (CUDA graph capture) */
/* The same with HOST buffers, synchronous: frames as in ofb_flow_pairs_host_ex (channels = 1: planar gray, 3: the
 * reference layout, channel 0 read; ofb_ctx_set_host_threads applies), through its sub-batch pipeline, so that uploads,
 * compute and downloads of different sub-batches overlap (pinned host memory makes the copies asynchronous; pageable
 * memory works too).  Each sub-batch runs what ofb_flow_pairs_fb_device runs; every output is bit-identical to that call
 * on the same frames.  fwd_total_h (n_pairs*h*w*2 floats) and status_h (n_pairs*h*w bytes) are required; bwd_total_h
 * (n_pairs*h*w*2 floats) and err2_h (n_pairs*h*w floats) may be NULL and are then not downloaded.  Arguments are checked as
 * there: p->flow_scale > 0, alpha >= 0, beta >= 0. */
int ofb_flow_pairs_fb_host(ofb_ctx *ctx, const ofb_params *p, const unsigned char *prev_h, const unsigned char *next_h,
                           int channels, float alpha, float beta, float *fwd_total_h, float *bwd_total_h, uint8_t *status_h,
                           float *err2_h);
/* The check on a frame sequence (ofb_stream): ofb_stream_push_bgr_host's upload, grayscale, optional bilateral filter and
 * pyramid of the new frame, then the flow previous->current and current->previous on the two pyramids the stream keeps,
 * the check and the downloads.  Every output is bit-identical to ofb_flow_pairs_fb_device on the two preprocessed frames.
 * fwd_total_h and status_h are required (h*w*2 floats, h*w bytes); flow_levels_h (forward residual flow, NULL or with NULL
 * entries as in ofb_flow_pairs_host_ex), bwd_total_h and err2_h may be NULL.  The first push only primes the pyramid
 * (*has_flow = 0, nothing written).  Pushes with and without the check may be mixed on one stream.  The backward level loop
 * runs on a second CUDA stream of the sequence, beside the forward one; the buffers of the backward direction, that
 * stream and its events are created by the first call (OFB_ERR_NOMEM, with the sequence left where it was, if the device
 * memory cannot be had), so a sequence that never runs the check uses no more device memory than before. */
int ofb_stream_push_bgr_host_fb(ofb_stream *s, const unsigned char *frame_bgr, float alpha, float beta,
                                float *const *flow_levels_h, float *fwd_total_h, float *bwd_total_h, uint8_t *status_h,
                                float *err2_h, int *has_flow);

/* ---- sparse pyramidal Lucas-Kanade: a list of points tracked through the pyramid; the reference has no counterpart ----
 * The KLT tracker (OpenCV's calcOpticalFlowPyrLK): each point is followed coarse to fine with several Gauss-Newton
 * iterations per level, on the pyramids of ofb_flow_pairs_device and with the dense path's derivative masks, bilinear rule
 * and solve.  Point p = (x, y) of pair b is in level-0 pixels; its flow d is in flow units (displacement s*d px,
 * s = p->flow_scale, as for the dense total flow).  Per point, in this order:
 *   x or y not finite, or outside [0, w-1] x [0, h-1]                -> OFB_PT_OUTSIDE, flow NaN, not tracked
 *   d = 0; for k = L-1 .. 0 (level k is (w>>k) x (h>>k)):
 *     PX = rint(x * (256 >> k)), PY = rint(y * (256 >> k))  (the float product is exact; rint rounds half to even)
 *     fields (exact integers, 0 outside the level): Ix = Dx (*) prev_k, Iy = Dy (*) prev_k, Sp = Dt (*) prev_k,
 *       Sn = Dt (*) next_k -- the reference's masks as correlations with zero padding (OptFlowGpu.cu:1040-1090)
 *     F@(X, Y), X, Y in 1/256 px: x0 = X >> 8, wx = X & 255 (arithmetic shift), likewise y0, wy; taps F00 = F(x0, y0),
 *       F01 = F(x0+1, y0), F10 = F(x0, y0+1), F11 = F(x0+1, y0+1);
 *       F@ = ((256-wy)*((256-wx)*F00 + wx*F01) + wy*((256-wx)*F10 + wx*F11) + 32768) >> 16   (the bilinear warp's rule)
 *     over the win x win offsets o = (ox, oy), |ox|, |oy| <= win/2: gx = Ix@(P + 256 o), gy = Iy@(P + 256 o),
 *       sp = Sp@(P + 256 o); a = sum gx*gx, dd = sum gy*gy, b = sum gx*gy (exact in int32: |gx|, |gy| <= 1020)
 *     min_eig > 0: lam < min_eig, lam = l1 / win^2 with l1 the smaller eigenvalue of [[a, b], [b, dd]], decided on the
 *       characteristic polynomial at mu = min_eig * win^2 (no square root, no division): in double, every operation
 *       rounded on its own, no fma, S = a + dd, mu = min_eig * (win^2) (both exact), det = a*dd - b*b exact in int64,
 *       then rounded to double; a window with det == 0 (lam = 0) is below every min_eig > 0.  Elsewhere the decision
 *       is that of the exact lam < min_eig except for min_eig within a relative 1e-6 of lam (the bound is reached
 *       only on near-isotropic windows, where the polynomial has a near-double root);
 *       mu > 0.5*S or det < mu * (S - mu)                                                     -> OFB_PT_LOW_TEXTURE, stop
 *     iterations i = 1 .. iters:
 *       !(|s*d.u| < 32768 && |s*d.v| < 32768) (float products)                                  -> OFB_PT_OUTSIDE, stop
 *       U = rint(d.u * s256), V = rint(d.v * s256), s256 = s * 256 (float; half to even)
 *       It(o) = Sn@(P + (U, V) + 256 o) - sp(o); tx = sum gx*It, ty = sum gy*It (exact in int32: |It| <= 3825, win <= 19)
 *       delta = the EXACT solve of (a, dd, b, tx, ty) (OFB_SOLVE_EXACT's operation order; the context's solve mode does
 *         not apply); d += delta (float adds)
 *       delta not finite (det == 0, Q3)                                                       -> OFB_PT_NONFINITE, stop
 *       eps > 0 and |s*delta.u| < eps and |s*delta.v| < eps (float products): the level is done
 *     d *= 2 unless k == 0
 *   A point that stopped at level k reports 2^k * d.  A point that ran through level 0 is OFB_PT_TRACKED, or OFB_PT_OUTSIDE
 *   with its flow kept when its final d fails the 32768 px test or its target (PX + U, PY + V) at level 0 lies outside
 *   [0, (w-1)*256] x [0, (h-1)*256].
 * With levels = 1, iters = 1, integer points and min_eig = 0 every sample is the field value itself and the solve is the
 * dense path's: the flow of a point is that of ofb_flow_pairs_device's coarsest level at that pixel, bit for bit.
 *   points_d: float2 (x, y), n_points per pair, pairs back to back (8-byte aligned); flow_d: the same shape (8-byte
 *   aligned); status_d: one byte per point.  p->warp_mode must be OFB_WARP_BILINEAR, p->flow_scale > 0 with s256 finite;
 *   1 <= n_points <= 2^24, 1 <= iters <= 64, eps and min_eig finite and >= 0; frames as in ofb_flow_pairs_device (at most
 *   65535 pairs).  Bad arguments are refused before anything is enqueued.  The pyramids live in the context workspace:
 *   ofb_ctx_reserve_pairs with the same parameters sizes it (CUDA graph capture).  With profiling on, the kernel gets an
 *   OFB_PROFILE_TRACK record and the pyramid build its OFB_PROFILE_PYRAMID record. */
#define OFB_PT_TRACKED 0
#define OFB_PT_NONFINITE 1
#define OFB_PT_LOW_TEXTURE 2
#define OFB_PT_OUTSIDE 3
int ofb_track_points_device(ofb_ctx *ctx, const ofb_params *p, const uint8_t *prev_d, const uint8_t *next_d,
                            size_t pitch_bytes, size_t image_stride_bytes, const float *points_d, int n_points,
                            int iters, float eps, float min_eig, float *flow_d, uint8_t *status_d, void *stream);

/* ---- Shi-Tomasi corners for the tracker: points to start from, found on the device; the reference has no counterpart ----
 * goodFeaturesToTrack's role with the tracker's own texture measure, so that a detected point is one the tracker accepts.
 * Images are planar u8 with the layout of ofb_flow_pairs_device (image i at img_d + i*image_stride_bytes), w x h each,
 * 1 <= n_images <= 65535, w * h < 2^31, odd win 3..19.
 * Score of pixel (x, y) (every pixel; ofb_min_eig_map_device writes it, n_images*h*w floats, tightly packed):
 *   gx = Dx (*) img, gy = Dy (*) img: the tracker's Ix, Iy at level 0 (Sobel correlations, 0 outside the frame; |g| <= 1020)
 *   over the win x win window centred on the pixel (field positions outside the frame contribute 0), exact in int32:
 *     A = sum gx^2, D = sum gy^2, B = sum gx*gy
 *   det = A*D - B*B, T = A - D, disc = T*T + 4*B*B exact in int64; S = A + D
 *   l1 = 0 if S == 0, else in double, every operation rounded to nearest on its own, no fma:
 *     l1 = (2.0 * (double)det) / ((double)S + sqrt((double)disc))     (the stable form of (S - sqrt(disc)) / 2)
 *   score = (float)(l1 / (double)(win*win))
 * This is the lam that ofb_track_points_device compares with min_eig: at an integer point with levels = 1 its a, dd, b are
 * A, D, B.
 * Detection, per image:
 *   interior: m <= x <= w-1-m and m <= y <= h-1-m, m = win/2 + 1 (every Sobel tap of the window lies inside the frame, so
 *     the zero padding cannot make corners); an image smaller than 2m+1 in either direction yields 0 corners
 *   thr = max(quality_level * max_score, min_score) (a float product), max_score the largest interior score; a pixel
 *     qualifies if score > thr (so a score of 0 never does)
 *   key order: p precedes q if score(p) > score(q), or the scores are equal and y_p*w + x_p < y_q*w + x_q
 *   candidates: qualifying interior pixels that precede each of their interior 8-neighbours (a strict local maximum in key
 *     order: a plateau yields one candidate per 3x3 neighbourhood, unlike OpenCV's score == dilate(score)); no two are
 *     8-adjacent, so an image has at most ceil(iw/2) * ceil(ih/2) of them (iw x ih the interior)
 *   selection: the candidates in key order; one is accepted unless an accepted corner lies at
 *     (double)(dx*dx + dy*dy) < (double)min_distance * (double)min_distance (dx, dy integer pixel differences, the sum
 *     exact in int64); stop after max_corners.  (OpenCV's sequential greedy; min_distance <= 1 suppresses nothing.)
 *   output: corners_d[i*max_corners + k] = (x, y) of the k-th accepted corner as floats, strongest first; scores_d
 *     (optional) its score; counts_d[i] the number accepted; the slots after it hold NaN (corners and scores), which the
 *     tracker reports OFB_PT_OUTSIDE: corners_d can be passed to ofb_track_points_device as its points.
 * Both calls are asynchronous on `stream` and never wait on the host (the counts stay on the device), so detection followed
 * by tracking can be captured as one CUDA graph after ofb_ctx_reserve_corners (and ofb_ctx_reserve_pairs) have sized the
 * workspace.  Limits: 1 <= max_corners <= 2^20, quality_level finite in [0, 1], min_distance and min_score finite and >= 0,
 * frames as in ofb_flow_pairs_device, corners_d 8-byte aligned, score_d / scores_d / counts_d 4-byte aligned; the
 * candidate slots n_images * ceil(iw/2) * ceil(ih/2) below 2^31 (OFB_ERR_UNSUPPORTED otherwise).  Bad arguments are
 * refused before anything is enqueued, the outputs untouched.  The detector's score map, candidates and cell grid live in
 * the context workspace.  With profiling on, each call gets one OFB_PROFILE_CORNERS record around its kernels. */
int ofb_min_eig_map_device(ofb_ctx *ctx, const uint8_t *img_d, size_t pitch_bytes, size_t image_stride_bytes, int w, int h,
                           int n_images, int win, float *score_d, void *stream);
int ofb_detect_corners_device(ofb_ctx *ctx, const uint8_t *img_d, size_t pitch_bytes, size_t image_stride_bytes, int w,
                              int h, int n_images, int win, int max_corners, float quality_level, float min_distance,
                              float min_score, float *corners_d, float *scores_d, int *counts_d, void *stream);
int ofb_ctx_reserve_corners(ofb_ctx *ctx, int w, int h, int n_images, int win, int max_corners);

/* Pinned host memory helpers for callers without a CUDA runtime of their own. */
int ofb_host_alloc(void **ptr, size_t bytes);
int ofb_host_free(void *ptr);

/* Number of kernels this library has launched on this context since creation (bench bookkeeping). */
int ofb_ctx_launch_count(const ofb_ctx *ctx, unsigned long long *count);

/* In-situ kernel timing for the roofline report.  While enabled, ofb_flow_pairs_device/_host put a
 * CUDA-event pair (on the stream the work is launched on) around every fused-LK launch, tagged with
 * its pyramid level, and around the pyramid build, tagged OFB_PROFILE_PYRAMID; the forward-backward entry points
 * also around the check kernel, tagged OFB_PROFILE_FB_CHECK, and ofb_track_points_device around its kernel, tagged
 * OFB_PROFILE_TRACK, and the corner entry points around their kernels, tagged OFB_PROFILE_CORNERS.  _enable(on) also
 * discards earlier records.  _read waits for the tagged events and returns their summed duration. */
#define OFB_PROFILE_PYRAMID 100
#define OFB_PROFILE_FB_CHECK 101
#define OFB_PROFILE_TRACK 102
#define OFB_PROFILE_CORNERS 103
int ofb_ctx_profile_enable(ofb_ctx *ctx, int on);
int ofb_ctx_profile_read(ofb_ctx *ctx, int tag, double *ms_sum, unsigned long long *n_records);

#ifdef __cplusplus
}
#endif
#endif /* OFB200_H */
