// ofb_common.cuh -- shared declarations of the sm_100a kernels and their launchers.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/ofb200.h"

namespace ofb {

// ---- error plumbing (ofb_api.cu) -----------------------------------------------------------
void set_error(const char *fmt, ...);
#define OFB_CUDA_TRY(expr)                                                                              \
    do {                                                                                                \
        cudaError_t _e = (expr);                                                                        \
        if (_e != cudaSuccess) {                                                                        \
            ofb::set_error("%s:%d: %s failed: %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
            return OFB_ERR_CUDA;                                                                        \
        }                                                                                               \
    } while (0)

// Makes `dev` current for the lifetime of the guard and restores the caller's device afterwards (every entry point of the
// C ABI uses it: a host that drives several GPUs from one thread keeps its own current device).
struct DeviceGuard {
    int prev = -1;
    bool ok = false;
    explicit DeviceGuard(int dev)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) {
            prev = -1;
            set_error("no usable CUDA device: %s", cudaGetErrorString(cudaGetLastError()));
            return;
        }
        if (prev != dev && cudaSetDevice(dev) != cudaSuccess) {
            set_error("cudaSetDevice(%d) failed: %s", dev, cudaGetErrorString(cudaGetLastError()));
            return;
        }
        ok = true;
    }
    ~DeviceGuard()
    {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

// ---- programmatic dependent launch (sm_90+) ------------------------------------------------------------------------------
// The kernels of a pair form a dependent chain (pyramid steps, then the levels coarse to fine), and for one pair or one
// strip each of them is short: launched this way a kernel may be scheduled while its predecessor in the stream is still
// draining -- its launch latency and prologue overlap the predecessor's tail -- and waits with pdl_wait() (before its first
// global-memory access) until the predecessor has completed and its memory is visible.  Every kernel launched through
// launch_pdl MUST call pdl_wait().  OFF by default (OFB_PDL=1 in the environment turns it on): measured on B200 the eager
// single-pair latency does not move (49.9 us either way), a replayed CUDA graph of one pair gets slower (43 -> 51 us) and so
// do row strips with several pairs in flight (0.247 -> 0.259 ms): early-scheduled CTAs hold SM slots while they wait.
bool pdl_enabled();
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
#endif

// ---- fused LK level (lk_level.cu) ----------------------------------------------------------
struct LkLevelArgs {
    const uint8_t *prev;   // planar u8, local rows [0, h_local)
    const uint8_t *next;
    size_t pitch;          // bytes, multiple of 16
    size_t image_stride;   // bytes between pairs, multiple of 16
    int w;                 // width
    int h_local;           // rows held by the buffers
    int y_off;             // global row of local row 0
    int h_global;          // height of the whole level
    int out_y0, out_y1;    // local rows to produce
    int n_pairs;
    int win;               // odd 3..19
    int warp_mode;         // OFB_WARP_*
    float flow_scale;
    const float *cum_in;   // coarser cumulative flow (float2), NULL => coarsest level, no warp
    int cum_w;             // coarser level width
    int cum_h_global;      // coarser level height (whole level)
    int cum_y_off;         // global coarse row of cum_in's row 0
    int cum_h_local;       // rows held by cum_in
    size_t cum_pair_stride;   // float2 elements between pairs
    // Composition on the fly (whole frames): cum_in is the RESIDUAL flow of the next-coarser level and cum2_in the cumulative
    // flow of the level above that ((cum_w >> 1) x (cum_h_global >> 1) per pair); NULL = cum_in is the cumulative flow itself
    const float *cum2_in;
    size_t cum2_pair_stride;  // float2 elements between pairs
    float *flow_out;       // float2, local rows (same origin as prev/next)
    float *cum_out;        // optional
    size_t flow_pair_stride;  // float2 elements between pairs (flow_out and cum_out)
    int *reach_overflow;   // optional device flag: a warp sample fell outside the local rows
    int sm_count;
    int solve_fast;        // OFB_SOLVE_FAST: tolerance-mode solve (lk_solve4_fast) instead of the bit-exact one
    // row strips, halo exchange fused into the kernel (strips.cu; zero = off)
    struct PeerPush {
        float *dst;            // neighbour's coarser-flow buffer, offset so that dst + 2*o is the peer's copy of this level's pixel o
        int row_lo, row_hi;    // local rows the neighbour needs
        unsigned *flag;        // arrival flag in the neighbour's memory
        const unsigned *done;  // in this rank's memory
    } push[2];
    int npush;
    struct PeerWait {
        const unsigned *flag;  // arrival flag in this rank's memory
        int crow_lo, crow_hi;  // local rows of cum_in the neighbour provides
    } wait[2];
    int nwait;
    unsigned *push_counter;    // [2], zero between launches
    const unsigned *epoch_src;
};
int launch_lk_level(const LkLevelArgs &a, cudaStream_t stream, unsigned long long *launches);
// The level's geometry and solve, everything else zero; callers add the coarser flow, cum_out and the peer fields.
// Whole frames: n_pairs images of w x h, every row produced.
LkLevelArgs lk_args_frame(const uint8_t *prev, const uint8_t *next, size_t pitch, size_t image_stride, int w, int h, int n_pairs,
                          int win, int warp_mode, float flow_scale, float *flow_out, int sm_count, int solve_fast);
// One row strip of one pair: rows [y_off, y_off + h_local) of a level of height h_global held, local rows
// [out_y0, out_y1) produced.
LkLevelArgs lk_args_strip(const uint8_t *prev, const uint8_t *next, size_t pitch, int w, int h_local, int y_off, int h_global,
                          int out_y0, int out_y1, int win, int warp_mode, float flow_scale, float *flow_out, int sm_count,
                          int solve_fast);
int preload_lk_level(int win); // loads the window's kernels now instead of at their first launch
int preload_pyramid();

// ---- pyramid (pyramid.cu) ------------------------------------------------------------------
int launch_pyr_down(const uint8_t *src, size_t src_pitch, size_t src_stride, int sw, int sh, uint8_t *dst,
                    size_t dst_pitch, size_t dst_stride, int n_images, int channels, cudaStream_t stream,
                    unsigned long long *launches, const uint8_t *src2 = nullptr, uint8_t *dst2 = nullptr);

int launch_pyr_roll(const uint8_t *src, size_t src_pitch, size_t src_stride, int sw, int sh, uint8_t *dst1, size_t pitch1,
                    size_t stride1, uint8_t *dst2, size_t pitch2, size_t stride2, int n_images, cudaStream_t stream,
                    unsigned long long *launches, const uint8_t *srcB = nullptr, uint8_t *dst1B = nullptr,
                    uint8_t *dst2B = nullptr, int sm_count = 0);

int launch_pyr_down_strip(const uint8_t *src, size_t src_pitch, int sw, int src_rows, int src_y_off, uint8_t *dst,
                          size_t dst_pitch, int dst_y0, int dst_y1, cudaStream_t stream, unsigned long long *launches,
                          int n_images = 1, size_t src_stride = 0, size_t dst_stride = 0);

// ---- stage kernels + layout helpers (stages.cu) --------------------------------------------
int launch_c3_to_planar(const uint8_t *src_c3, int w, int h, int n_images, uint8_t *dst, size_t dst_pitch,
                        size_t dst_stride, cudaStream_t stream, unsigned long long *launches);
int launch_conv_c3_f32(const uint8_t *src_c3, int w, int h, float *dst, const float *mask_host, int mw, int mh,
                       cudaStream_t stream, unsigned long long *launches);
int launch_conv_c3_u8(const uint8_t *src_c3, int w, int h, uint8_t *dst, const float *mask_host, int mw, int mh,
                      cudaStream_t stream, unsigned long long *launches);
int launch_debug_view(const uint8_t *prev_c3, const uint8_t *cur_c3, int w, int h, int k, int which, uint8_t *out,
                      cudaStream_t stream, unsigned long long *launches);
int launch_srm_f32(const float *a, const float *b, int w, int h, int ww, int wh, float *dst, cudaStream_t stream,
                   unsigned long long *launches);
int launch_inverse_f32(const float *sxx, const float *syy, const float *sxy, const float *sxt, const float *syt,
                       float *flow, int n, cudaStream_t stream, unsigned long long *launches);
int launch_compose_cum(const float *flow_k, const float *cum_coarser, int w, int h, int n_pairs, float *cum_out,
                       cudaStream_t stream, unsigned long long *launches);

// ---- forward-backward consistency check (fb_check.cu) ---------------------------------------
int launch_fb_check(const float *fwd, const float *bwd, int w, int h, int n_pairs, float flow_scale, float alpha, float beta,
                    uint8_t *status, float *err2, cudaStream_t stream, unsigned long long *launches);
// row strips (strips.cu): own rows [y0, y0 + rows) against backward rows [b0, b1); bit 2 of *flag for UNCHECKED pixels
int launch_fb_check_strip(const float *fwd, const float *bwd_rows, int w, int h, int y0, int rows, int b0, int b1, float flow_scale,
                          float alpha, float beta, uint8_t *status, float *err2, int *flag, cudaStream_t stream,
                          unsigned long long *launches);
int preload_fb_check_strip();

// ---- sparse pyramidal LK, points tracked through the pyramid (track.cu) -------------------------------
struct TrackArgs {
    const uint8_t *prev[OFB_MAX_LEVELS], *next[OFB_MAX_LEVELS]; // level k of pair 0; pair i at + i * istr[k]
    size_t pitch[OFB_MAX_LEVELS], istr[OFB_MAX_LEVELS];
    int w, h, levels;          // level 0 size; level k is (w >> k) x (h >> k)
    int n_pairs, n_points;     // points per pair
    const float *points;       // float2 (x, y) in level-0 pixels, n_pairs * n_points
    float *flow;               // float2, n_pairs * n_points
    uint8_t *status;           // OFB_PT_*, n_pairs * n_points
    int iters;
    float eps, min_eig, flow_scale;
};
int launch_track_points(const TrackArgs &a, int win, cudaStream_t stream, unsigned long long *launches);

// ---- Shi-Tomasi corners for the tracker (corners.cu) ---------------------------------------------------------------
struct CornerArgs {
    const uint8_t *img;  // image i at img + i * istr
    size_t pitch, istr;
    int w, h, n;
    int m;               // interior margin win/2 + 1
    float *map;          // score of image i at map + i * map_stride, rows of w floats
    size_t map_stride;
    unsigned *max_bits;  // optional: per image, the float bits of the interior maximum (zeroed before the launch)
};
int launch_corner_score(const CornerArgs &a, int win, cudaStream_t stream, unsigned long long *launches);
struct CornerPlan {
    int m, iw, ih;       // interior margin and size (0 when the image has no interior)
    long long cap;       // candidate slots per image: ceil(iw/2) * ceil(ih/2)
    long long total;     // cap * n
};
void plan_corners(int w, int h, int n, int win, CornerPlan *p);
int corner_sort_bytes(long long total, int n, size_t *bytes); // temporary storage of the per-image sort
struct DetectArgs {
    CornerPlan plan;
    const uint8_t *img;
    size_t pitch, istr;
    int w, h, n, max_corners;
    float quality_level, min_distance, min_score;
    // workspace
    float *map;                              // n * h * w
    unsigned *max_bits;                      // n
    int *seg_begin, *seg_end;                // n each
    unsigned long long *keys_in, *keys_out;  // plan.total each
    int *grid;                               // n * iw * ih (the finest cell grid)
    void *sort_tmp;
    size_t sort_bytes;
    // outputs
    float *corners, *scores;
    int *counts;
};
int launch_detect_corners(const DetectArgs &d, int win, cudaStream_t stream, unsigned long long *launches);

int launch_grayscale(const uint8_t *src_c3, int w, int h, uint8_t *dst_c3, uint8_t *dst_planar, size_t dst_pitch,
                     cudaStream_t stream, unsigned long long *launches);
int launch_bilateral(const uint8_t *src, const uint8_t *gray, size_t pitch, int channels, int w, int h, int ww, int wh,
                     double sigmaS, double sigmaB, double *lut_dev, uint8_t *dst, size_t dst_pitch, cudaStream_t stream,
                     unsigned long long *launches);

// cuTensorMapEncodeTiled resolved through the runtime (no link-time libcuda dependency).
typedef CUresult (*PFN_encodeTiled)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                    const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
PFN_encodeTiled get_encode_tiled();

} // namespace ofb
