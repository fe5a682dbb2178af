// ofb_api.cu -- context object and the extern "C" surface declared in include/ofb200.h.
#include "host_extract.hpp"
#include "ofb_common.cuh"

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

namespace ofb {

static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

} // namespace ofb

#define OFB_LANES 6 /* streams available to the batched host entry point; it uses c->lanes of them */

// One growable device workspace per context; carved by offset for each call.  Growing it frees the
// old block (cudaFree synchronises the device), so steady-state calls allocate nothing -- unlike
// the reference, which does 30 cudaMalloc/cudaFree pairs per level (OptFlowGpu.cu:1105-1124 etc.).
struct ofb_ctx {
    int device = 0;
    int sm_count = 0;
    int lanes = 3;      // sub-batches in flight in ofb_flow_pairs_host (developer override: OFB_E2E_LANES)
    int sub_pairs = 0;  // pairs per sub-batch there; 0 = chosen from the batch size (developer override: OFB_E2E_SUB)
    int solve_fast = 0; // OFB_SOLVE_*: which 2x2 solve the fused level kernel runs (ofb_ctx_set_solve)
    cudaStream_t stream = nullptr; // used by the synchronous host-pointer entry points
    cudaStream_t lane_stream[OFB_LANES] = {}; // the batched host entry point pipelines sub-batches over these
    uint8_t *ws = nullptr;
    size_t ws_bytes = 0;
    // The workspace serves ONE stream at a time: every asynchronous use records ws_event on its stream, and a later user
    // on another stream waits for it first (ws_acquire / ws_release).
    cudaEvent_t ws_event = nullptr;
    cudaStream_t ws_stream = nullptr;
    bool ws_busy = false;
    unsigned long long launches = 0;
    // optional in-situ timing: CUDA events around each fused-LK launch (tag = level) and around the
    // pyramid build (tag = OFB_PROFILE_PYRAMID), recorded on the stream the work is launched on
    struct ProfRec {
        int tag;
        cudaEvent_t a, b;
    };
    double *bil_lut = nullptr; // range-weight table of the bilateral pre-filter (device)
    // 3-channel host images: channel 0 extracted by host threads into pinned planar staging buffers, one pair of buffers
    // per lane (ofb_ctx_set_host_threads; 0 = all three channels are uploaded and the device drops two)
    int host_threads = 0;
    ofb::HostPool *pool = nullptr;
    uint8_t *stage = nullptr;
    size_t stage_bytes = 0;
    cudaEvent_t stage_ev[OFB_LANES] = {};
    bool prof_on = false;
    std::vector<ProfRec> prof;
};

namespace ofb {

// accessors for the other translation units (strips.cu): ofb_ctx stays private to this file
int ctx_device(const ofb_ctx *c) { return c->device; }
int ctx_sm_count(const ofb_ctx *c) { return c->sm_count; }
int ctx_solve_fast(const ofb_ctx *c) { return c->solve_fast; }
unsigned long long *ctx_launch_counter(ofb_ctx *c) { return &c->launches; }

// Growing frees the old block after a device synchronisation: CUDA graphs captured from earlier calls hold pointers
// into it and must be re-captured (ofb_ctx_reserve_pairs sizes the workspace up front so that this never happens).
static int ws_reserve(ofb_ctx *c, size_t bytes)
{
    if (bytes <= c->ws_bytes) return OFB_OK;
    if (c->ws) {
        OFB_CUDA_TRY(cudaDeviceSynchronize());
        OFB_CUDA_TRY(cudaFree(c->ws));
        c->ws = nullptr;
        c->ws_bytes = 0;
    }
    const size_t want = align_up(bytes + bytes / 8, 1 << 20);
    cudaError_t e = cudaMalloc(reinterpret_cast<void **>(&c->ws), want);
    if (e != cudaSuccess) {
        set_error("workspace cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
        cudaGetLastError();
        return OFB_ERR_NOMEM;
    }
    c->ws_bytes = want;
    return OFB_OK;
}

// Orders the uses of the shared workspace across streams (see ofb_ctx::ws_event).
// A stream that is being captured into a CUDA graph takes no part: a capture cannot depend on eager work of another
// stream, and an event recorded inside a capture belongs to the graph.  Replays of such a graph are ordered against the
// context's other users by their caller (one context per concurrently used stream is the simple rule).
static bool ws_capturing(cudaStream_t st)
{
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    return cudaStreamIsCapturing(st, &cap) == cudaSuccess && cap != cudaStreamCaptureStatusNone;
}
static int ws_acquire(ofb_ctx *c, cudaStream_t st)
{
    if (c->ws_busy && c->ws_stream != st && !ws_capturing(st)) OFB_CUDA_TRY(cudaStreamWaitEvent(st, c->ws_event, 0));
    return OFB_OK;
}
static int ws_release(ofb_ctx *c, cudaStream_t st)
{
    if (ws_capturing(st)) return OFB_OK;
    OFB_CUDA_TRY(cudaEventRecord(c->ws_event, st));
    c->ws_stream = st;
    c->ws_busy = true;
    return OFB_OK;
}

struct Carver {
    size_t off = 0;
    size_t take(size_t bytes)
    {
        const size_t o = off;
        off = align_up(off + bytes, 256);
        return o;
    }
};

static int check_params(const ofb_params *p)
{
    if (!p) {
        set_error("params is NULL");
        return OFB_ERR_INVALID;
    }
    if (p->levels < 1 || p->levels > OFB_MAX_LEVELS) {
        set_error("levels %d outside 1..%d", p->levels, OFB_MAX_LEVELS);
        return OFB_ERR_INVALID;
    }
    if (p->w < 1 || p->h < 1 || (p->w >> (p->levels - 1)) < 2 || (p->h >> (p->levels - 1)) < 2) {
        set_error("frame %dx%d too small for %d levels (coarsest level must be at least 2x2)", p->w, p->h, p->levels);
        return OFB_ERR_INVALID;
    }
    if (p->win < 3 || p->win > OFB_MAX_WINDOW || !(p->win & 1)) {
        set_error("window %d not supported (odd 3..%d)", p->win, OFB_MAX_WINDOW);
        return OFB_ERR_UNSUPPORTED;
    }
    if (p->warp_mode < OFB_WARP_AS_WRITTEN || p->warp_mode > OFB_WARP_BILINEAR) {
        set_error("unknown warp mode %d", p->warp_mode);
        return OFB_ERR_INVALID;
    }
    if (p->n_pairs < 1) {
        set_error("n_pairs %d < 1", p->n_pairs);
        return OFB_ERR_INVALID;
    }
    return OFB_OK;
}

// Pyramids of both frames + coarse-to-fine LK, everything device resident.  `base` is the
// context workspace region reserved for this call.
struct PairPlan {
    size_t pitch[OFB_MAX_LEVELS], istride[OFB_MAX_LEVELS];
    size_t off_prev[OFB_MAX_LEVELS], off_next[OFB_MAX_LEVELS], off_cum[OFB_MAX_LEVELS];
    size_t bytes = 0;
};

// Two pyramid steps per launch (pyramid.cu: pyr_roll_kernel<true>); OFB_PYR_FUSE=0 builds level by level (A/B measurements).
static bool pyr_fuse_enabled()
{
    static const bool on = [] {
        const char *e = getenv("OFB_PYR_FUSE");
        return !(e && e[0] == '0');
    }();
    return on;
}

static void plan_pairs(const ofb_params *p, PairPlan *pl, Carver *cv)
{
    for (int k = 0; k < p->levels; k++) {
        const int wk = p->w >> k, hk = p->h >> k;
        pl->pitch[k] = align_up((size_t)wk, 64);
        pl->istride[k] = pl->pitch[k] * (size_t)hk;
        pl->off_prev[k] = pl->off_next[k] = pl->off_cum[k] = (size_t)-1;
        if (k >= 1) {
            pl->off_prev[k] = cv->take(pl->istride[k] * p->n_pairs);
            pl->off_next[k] = cv->take(pl->istride[k] * p->n_pairs);
        }
        if (k >= 1 && k <= p->levels - 2) pl->off_cum[k] = cv->take((size_t)wk * hk * 8 * p->n_pairs);
    }
    pl->bytes = cv->off;
}

static int prof_begin(ofb_ctx *c, int tag, cudaStream_t st)
{
    if (!c->prof_on) return OFB_OK;
    ofb_ctx::ProfRec r{tag, nullptr, nullptr};
    OFB_CUDA_TRY(cudaEventCreate(&r.a));
    OFB_CUDA_TRY(cudaEventCreate(&r.b));
    OFB_CUDA_TRY(cudaEventRecord(r.a, st));
    c->prof.push_back(r);
    return OFB_OK;
}
static int prof_end(ofb_ctx *c, cudaStream_t st)
{
    if (!c->prof_on || c->prof.empty()) return OFB_OK;
    OFB_CUDA_TRY(cudaEventRecord(c->prof.back().b, st));
    return OFB_OK;
}

// Level-0 frames and the pyramid levels built from them, both frames of every pair.
struct PairLevels {
    const uint8_t *prev[OFB_MAX_LEVELS], *next[OFB_MAX_LEVELS];
    size_t pitch[OFB_MAX_LEVELS], istr[OFB_MAX_LEVELS];
};

// Levels 1..L-1 of one image set (b == NULL) or two, n images of w x h each, from their level 0, with the
// OFB_PROFILE_PYRAMID record: one launch per one or two pyramid steps, both sets in it when the grid allows.
static int build_pyramid_levels(ofb_ctx *c, int w, int h, int L, const uint8_t *const *a, const uint8_t *const *b,
                                const size_t *pitch, const size_t *istr, int n, cudaStream_t st)
{
    if (L < 2) return OFB_OK;
    int rc = prof_begin(c, OFB_PROFILE_PYRAMID, st);
    if (rc) return rc;
    const bool joint = b && 2 * n <= 65535; // grid.z limit: both sets in one launch
    auto lv = [](const uint8_t *const *set, int k) { return const_cast<uint8_t *>(set[k]); };
    for (int k = 1; k < L;) {
        // two pyramid steps per launch where two are left (level k is then never read back), else one
        const bool two = pyr_fuse_enabled() && k + 1 < L;
        for (int f = 0; f < (b && !joint ? 2 : 1); f++) {
            const uint8_t *const *src = f ? b : a;
            rc = launch_pyr_roll(src[k - 1], pitch[k - 1], istr[k - 1], w >> (k - 1), h >> (k - 1), lv(src, k), pitch[k], istr[k],
                                 two ? lv(src, k + 1) : nullptr, two ? pitch[k + 1] : 0, two ? istr[k + 1] : 0, n, st, &c->launches,
                                 joint ? b[k - 1] : nullptr, joint ? lv(b, k) : nullptr, joint && two ? lv(b, k + 1) : nullptr,
                                 c->sm_count);
            if (rc) return rc;
        }
        k += two ? 2 : 1;
    }
    return prof_end(c, st);
}

// Pyramids of both frames: levels 1..L-1 into the plan's regions of `base`.
static int build_pyramids(ofb_ctx *c, const ofb_params *p, const PairPlan &pl, uint8_t *base, const uint8_t *prev0,
                          const uint8_t *next0, size_t pitch0, size_t istride0, PairLevels *lv, cudaStream_t st)
{
    lv->prev[0] = prev0;
    lv->next[0] = next0;
    lv->pitch[0] = pitch0;
    lv->istr[0] = istride0;
    for (int k = 1; k < p->levels; k++) {
        lv->prev[k] = base + pl.off_prev[k];
        lv->next[k] = base + pl.off_next[k];
        lv->pitch[k] = pl.pitch[k];
        lv->istr[k] = pl.istride[k];
    }
    return build_pyramid_levels(c, p->w, p->h, p->levels, lv->prev, lv->next, lv->pitch, lv->istr, p->n_pairs, st);
}

// The coarse-to-fine loop of main.cu:256-262 on built pyramids, prev -> next or (backward) next -> prev; cum[k]
// (k = 1..L-2) are the regions where warped levels materialise their cumulative flow.
static int run_levels(ofb_ctx *c, const ofb_params *p, const PairLevels &lv, bool backward, float *const *flow_levels,
                      float *const *cum, float *total_flow, cudaStream_t st)
{
    const int L = p->levels, n = p->n_pairs;
    const uint8_t *const *pp = backward ? lv.next : lv.prev, *const *pn = backward ? lv.prev : lv.next;
    auto W = [p](int k) { return p->w >> k; };
    auto H = [p](int k) { return p->h >> k; };
    // Which warped levels materialise their cumulative flow.  Level 1 need not when level 0 composes it on the fly from
    // flow_1 and cum_2 (lk_level_kernel<..., COMP>): 8 bytes per pixel less to write at level 1, whose kernel is bound by
    // exactly those stores.  Composition needs even sizes (no clamped coarse indices), TMA-able rows and a per-pixel warp
    // mode.  Only level 0 composes, and only when it does not itself write the total flow: a reader that also writes its
    // cumulative flow pays more for the composition than the (four times smaller) coarser level saves -- measured on the
    // 4-level 4K configuration: level 1 +8 %, level 2 -20 %, a net loss.
    bool mat[OFB_MAX_LEVELS] = {}, comp[OFB_MAX_LEVELS] = {};
    for (int k = 1; k < L; k++) mat[k] = true;
    static const bool allow_compose = [] {
        const char *e = getenv("OFB_NO_COMPOSE"); // developer switch for A/B measurements
        return !(e && e[0] == '1');
    }();
    if (L >= 3 && !total_flow && allow_compose && p->warp_mode != OFB_WARP_AS_WRITTEN) {
        const bool even = !((W(0) | H(0) | W(1) | H(1) | W(2)) & 1);
        const float *c2 = (2 == L - 1) ? flow_levels[2] : cum[2];
        const bool aligned = !((reinterpret_cast<uintptr_t>(flow_levels[1]) | reinterpret_cast<uintptr_t>(c2)) & 15);
        if (even && aligned) {
            comp[0] = true;
            mat[1] = false;
        }
    }
    for (int k = L - 1; k >= 0; k--) {
        LkLevelArgs a = lk_args_frame(pp[k], pn[k], lv.pitch[k], lv.istr[k], W(k), H(k), n, p->win, p->warp_mode, p->flow_scale,
                                      flow_levels[k], c->sm_count, c->solve_fast);
        if (k < L - 1) {
            // cum_{k+1}: the coarsest level's cumulative flow is its residual flow; a level that did not materialise its
            // own hands over its residual flow together with its parent's cumulative flow
            a.cum_in = (k + 1 == L - 1 || comp[k]) ? flow_levels[k + 1] : cum[k + 1];
            a.cum_w = W(k + 1);
            a.cum_h_global = H(k + 1);
            a.cum_y_off = 0;
            a.cum_h_local = H(k + 1);
            a.cum_pair_stride = (size_t)W(k + 1) * H(k + 1);
            if (comp[k]) {
                a.cum2_in = (k + 2 == L - 1) ? flow_levels[k + 2] : cum[k + 2];
                a.cum2_pair_stride = (size_t)W(k + 2) * H(k + 2);
            }
        }
        if (k == 0) a.cum_out = total_flow;
        else if (k <= L - 2 && mat[k]) a.cum_out = cum[k];
        int rc = prof_begin(c, k, st);
        if (rc) return rc;
        rc = launch_lk_level(a, st, &c->launches);
        if (rc) return rc;
        rc = prof_end(c, st);
        if (rc) return rc;
    }
    return OFB_OK;
}

// ofb_flow_pairs_device and the batched host entry point: both pyramids, then the level loop.
static int run_pairs_device(ofb_ctx *c, const ofb_params *p, const PairPlan &pl, uint8_t *base, const uint8_t *prev0,
                            const uint8_t *next0, size_t pitch0, size_t istride0, float *const *flow_levels,
                            float *total_flow, cudaStream_t st)
{
    PairLevels lv;
    int rc = build_pyramids(c, p, pl, base, prev0, next0, pitch0, istride0, &lv, st);
    if (rc) return rc;
    float *cum[OFB_MAX_LEVELS] = {};
    for (int k = 1; k <= p->levels - 2; k++) cum[k] = reinterpret_cast<float *>(base + pl.off_cum[k]);
    return run_levels(c, p, lv, false, flow_levels, cum, total_flow, st);
}

// Workspace of the forward-backward call: the regions of plan_pairs (both pyramids, the forward direction's cumulative
// flow), then the residual flow of every level of both directions and the backward direction's cumulative flow.
struct PairFbPlan {
    PairPlan pl;
    size_t off_flow[2][OFB_MAX_LEVELS], off_cum_b[OFB_MAX_LEVELS];
    size_t bytes = 0;
};

static void plan_pairs_fb(const ofb_params *p, PairFbPlan *fp)
{
    Carver cv;
    plan_pairs(p, &fp->pl, &cv);
    auto bytes = [p](int k) { return (size_t)(p->w >> k) * (p->h >> k) * 8 * p->n_pairs; };
    for (int d = 0; d < 2; d++)
        for (int k = 0; k < p->levels; k++) fp->off_flow[d][k] = cv.take(bytes(k));
    for (int k = 0; k < p->levels; k++) {
        fp->off_cum_b[k] = (size_t)-1;
        if (k >= 1 && k <= p->levels - 2) fp->off_cum_b[k] = cv.take(bytes(k));
    }
    fp->bytes = cv.off;
}

// The frames of the device entry points: `ptrs_ok` (their non-NULL pointers, `null_msg` otherwise), pitch, image stride,
// and the pair count, before the workspace grows or anything is enqueued: the level kernels and the check take at most
// 65535 pairs.
static int check_device_frames(const ofb_params *p, bool ptrs_ok, const char *null_msg, size_t pitch_bytes,
                               size_t image_stride_bytes)
{
    if (!ptrs_ok) {
        set_error("%s", null_msg);
        return OFB_ERR_INVALID;
    }
    if (pitch_bytes < (size_t)p->w || (p->n_pairs > 1 && image_stride_bytes < pitch_bytes * (size_t)p->h)) {
        set_error("pitch %zu / image stride %zu too small for %dx%d", pitch_bytes, image_stride_bytes, p->w, p->h);
        return OFB_ERR_INVALID;
    }
    if (p->n_pairs > 65535) {
        set_error("at most 65535 pairs per call (got %d)", p->n_pairs);
        return OFB_ERR_INVALID;
    }
    return OFB_OK;
}

static int check_fb_args(float flow_scale, float alpha, float beta)
{
    if (!(std::isfinite(flow_scale) && flow_scale > 0.0f)) {
        set_error("flow_scale %g must be finite and > 0", (double)flow_scale);
        return OFB_ERR_INVALID;
    }
    if (!(std::isfinite(alpha) && alpha >= 0.0f && std::isfinite(beta) && beta >= 0.0f)) {
        set_error("alpha %g / beta %g must be finite and >= 0", (double)alpha, (double)beta);
        return OFB_ERR_INVALID;
    }
    return OFB_OK;
}

static int check_fb_buffers(const float *fwd, const float *bwd, const uint8_t *status, const float *err2)
{
    if (!fwd || !bwd || !status) {
        set_error("NULL flow or status pointer");
        return OFB_ERR_INVALID;
    }
    if (((reinterpret_cast<uintptr_t>(fwd) | reinterpret_cast<uintptr_t>(bwd)) & 7) || (reinterpret_cast<uintptr_t>(err2) & 3)) {
        set_error("flow fields must be 8-byte aligned, err2 4-byte aligned");
        return OFB_ERR_INVALID;
    }
    return OFB_OK;
}

// The check kernel with its OFB_PROFILE_FB_CHECK record.
static int run_fb_check(ofb_ctx *c, const float *fwd, const float *bwd, int w, int h, int n_pairs, float flow_scale, float alpha,
                        float beta, uint8_t *status, float *err2, cudaStream_t st)
{
    int rc = prof_begin(c, OFB_PROFILE_FB_CHECK, st);
    if (rc) return rc;
    if ((rc = launch_fb_check(fwd, bwd, w, h, n_pairs, flow_scale, alpha, beta, status, err2, st, &c->launches))) return rc;
    return prof_end(c, st);
}

// The device-side body of ofb_flow_pairs_fb_device and ofb_flow_pairs_fb_host: both pyramids once, the level loop
// prev->next and then next->prev on them, the check.  `base` holds the regions of `fp`.
static int run_pairs_fb_device(ofb_ctx *c, const ofb_params *p, const PairFbPlan &fp, uint8_t *base, const uint8_t *prev0,
                               const uint8_t *next0, size_t pitch0, size_t istride0, float alpha, float beta, float *fwd_total,
                               float *bwd_total, uint8_t *status, float *err2, cudaStream_t st)
{
    PairLevels lv;
    int rc = build_pyramids(c, p, fp.pl, base, prev0, next0, pitch0, istride0, &lv, st);
    if (rc) return rc;
    float *flow[2][OFB_MAX_LEVELS], *cum[2][OFB_MAX_LEVELS] = {};
    for (int k = 0; k < p->levels; k++) {
        for (int d = 0; d < 2; d++) flow[d][k] = reinterpret_cast<float *>(base + fp.off_flow[d][k]);
        if (k >= 1 && k <= p->levels - 2) {
            cum[0][k] = reinterpret_cast<float *>(base + fp.pl.off_cum[k]);
            cum[1][k] = reinterpret_cast<float *>(base + fp.off_cum_b[k]);
        }
    }
    if ((rc = run_levels(c, p, lv, false, flow[0], cum[0], fwd_total, st))) return rc;
    if ((rc = run_levels(c, p, lv, true, flow[1], cum[1], bwd_total, st))) return rc;
    return run_fb_check(c, fwd_total, bwd_total, p->w, p->h, p->n_pairs, p->flow_scale, alpha, beta, status, err2, st);
}

// One sub-batch of the batched host entry points: pairs [first, first + p.n_pairs) of the call, whose level-0 frames have
// been uploaded into prev0 / next0 inside the lane's workspace region B; its work goes on the lane's stream st.
struct HostSub {
    ofb_params p;
    int first;
    uint8_t *B;
    const uint8_t *prev0, *next0;
    size_t pitch0, istride0;
    cudaStream_t st;
};

// The sub-batch pipeline of the batched host entry points (ofb_flow_pairs_host / _ex and ofb_flow_pairs_fb_host), with
// host input in the layout of `channels`.  plan_lane(sub, &cv) lays out the caller's regions of a lane's workspace after the
// level-0 frames and returns the lane's end offset; run_sub(HostSub) enqueues a sub-batch's compute and downloads.
template <class PlanLane, class RunSub>
static int host_pipeline(ofb_ctx *c, const ofb_params *p, const unsigned char *prev_h, const unsigned char *next_h, int channels,
                         PlanLane plan_lane, RunSub run_sub)
{
    // Software pipeline over sub-batches on OFB_LANES streams: while one lane downloads its flow the
    // other uploads and computes, so the PCIe directions and the SMs overlap (with pinned host memory).
    // Sub-batches are kept small (at least eight per lane when the batch allows): the first upload and the last
    // download are the part of the pipeline nothing overlaps, and a 1080p pair already is 12 MB in and 22 MB out.
    const int n = p->n_pairs;
    const int LANES = c->lanes;
    int sub = n / (8 * LANES);
    if (sub < 1) sub = 1;
    if (sub > 8) sub = 8;
    if (c->sub_pairs > 0) sub = c->sub_pairs < n ? c->sub_pairs : n;
    const size_t pitch0 = align_up((size_t)p->w, 64), istride0 = pitch0 * (size_t)p->h;
    const size_t c3 = (size_t)p->w * p->h * 3;
    size_t lane_bytes = 0;
    size_t off_p0, off_n0, off_c3 = 0;
    {
        Carver cv;
        off_p0 = cv.take(istride0 * sub);
        off_n0 = cv.take(istride0 * sub);
        if (channels == 3) off_c3 = cv.take(c3 * sub * 2);
        lane_bytes = align_up(plan_lane(sub, &cv), 256);
    }
    int rc = ws_reserve(c, lane_bytes * LANES);
    if (rc) return rc;
    // 3-channel input with host threads: channel 0 is extracted on the host into pinned planar staging buffers (one
    // prev + one next buffer per lane) and only those bytes are uploaded (host_extract.cpp)
    const bool host_extract = channels == 3 && c->host_threads > 0;
    const size_t frame_px = (size_t)p->w * p->h, stage_lane = 2 * frame_px * sub;
    bool stage_used[OFB_LANES] = {};
    if (host_extract) {
        if (!c->pool) {
            try {
                c->pool = new ofb::HostPool(c->host_threads);
            } catch (...) {
                set_error("flow_pairs_host: could not start %d host threads", c->host_threads);
                return OFB_ERR_NOMEM;
            }
        }
        if (c->stage_bytes < stage_lane * LANES) {
            if (c->stage) OFB_CUDA_TRY(cudaFreeHost(c->stage));
            c->stage = nullptr;
            c->stage_bytes = 0;
            OFB_CUDA_TRY(cudaHostAlloc(reinterpret_cast<void **>(&c->stage), stage_lane * LANES, cudaHostAllocDefault));
            c->stage_bytes = stage_lane * LANES;
        }
        for (int lane = 0; lane < LANES; lane++)
            if (!c->stage_ev[lane]) OFB_CUDA_TRY(cudaEventCreateWithFlags(&c->stage_ev[lane], cudaEventDisableTiming));
    }
    for (int lane = 0; lane < LANES; lane++)
        if ((rc = ws_acquire(c, c->lane_stream[lane]))) return rc;
    for (int first = 0, sb = 0; first < n; first += sub, sb++) {
        const int lane = sb % LANES;
        const int cnt = (n - first < sub) ? n - first : sub;
        cudaStream_t st = c->lane_stream[lane];
        uint8_t *B = c->ws + lane_bytes * lane;
        if (channels == 1) {
            OFB_CUDA_TRY(cudaMemcpy2DAsync(B + off_p0, pitch0, prev_h + (size_t)first * p->w * p->h, (size_t)p->w, (size_t)p->w,
                                           (size_t)p->h * cnt, cudaMemcpyHostToDevice, st));
            OFB_CUDA_TRY(cudaMemcpy2DAsync(B + off_n0, pitch0, next_h + (size_t)first * p->w * p->h, (size_t)p->w, (size_t)p->w,
                                           (size_t)p->h * cnt, cudaMemcpyHostToDevice, st));
        } else if (host_extract) {
            uint8_t *sp = c->stage + stage_lane * lane, *sn = sp + frame_px * sub;
            if (stage_used[lane]) OFB_CUDA_TRY(cudaEventSynchronize(c->stage_ev[lane])); // the lane's previous upload has left the buffers
            ofb::c3_extract_pair_sets(c->pool, prev_h + c3 * first, next_h + c3 * first, sp, sn, frame_px * cnt);
            OFB_CUDA_TRY(cudaMemcpy2DAsync(B + off_p0, pitch0, sp, (size_t)p->w, (size_t)p->w, (size_t)p->h * cnt,
                                           cudaMemcpyHostToDevice, st));
            OFB_CUDA_TRY(cudaMemcpy2DAsync(B + off_n0, pitch0, sn, (size_t)p->w, (size_t)p->w, (size_t)p->h * cnt,
                                           cudaMemcpyHostToDevice, st));
            OFB_CUDA_TRY(cudaEventRecord(c->stage_ev[lane], st));
            stage_used[lane] = true;
        } else {
            OFB_CUDA_TRY(cudaMemcpyAsync(B + off_c3, prev_h + c3 * first, c3 * cnt, cudaMemcpyHostToDevice, st));
            OFB_CUDA_TRY(cudaMemcpyAsync(B + off_c3 + c3 * sub, next_h + c3 * first, c3 * cnt, cudaMemcpyHostToDevice, st));
            rc = launch_c3_to_planar(B + off_c3, p->w, p->h, cnt, B + off_p0, pitch0, istride0, st, &c->launches);
            if (rc) return rc;
            rc = launch_c3_to_planar(B + off_c3 + c3 * sub, p->w, p->h, cnt, B + off_n0, pitch0, istride0, st, &c->launches);
            if (rc) return rc;
        }
        HostSub s{*p, first, B, B + off_p0, B + off_n0, pitch0, istride0, st};
        s.p.n_pairs = cnt;
        if ((rc = run_sub(s))) return rc;
    }
    for (int lane = 0; lane < LANES; lane++) OFB_CUDA_TRY(cudaStreamSynchronize(c->lane_stream[lane]));
    return OFB_OK;
}

} // namespace ofb

using namespace ofb;

#define OFB_CHECK_CTX(c)                     \
    do {                                     \
        if (!(c)) {                          \
            set_error("context is NULL");    \
            return OFB_ERR_INVALID;          \
        }                                    \
    } while (0)
#define OFB_GUARD(c)            \
    DeviceGuard _guard((c)->device); \
    if (!_guard.ok) return OFB_ERR_CUDA

extern "C" {

const char *ofb_last_error(void) { return g_err; }
int ofb_version(void) { return 101; }

int ofb_ctx_create(int device, ofb_ctx **out)
{
    if (!out) {
        set_error("out is NULL");
        return OFB_ERR_INVALID;
    }
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev < 1) {
        set_error("no CUDA device available (%s); this library has no CPU fallback",
                  e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
        cudaGetLastError();
        return OFB_ERR_CUDA;
    }
    if (device < 0 || device >= ndev) {
        set_error("device %d outside 0..%d", device, ndev - 1);
        return OFB_ERR_INVALID;
    }
    DeviceGuard g(device);
    if (!g.ok) return OFB_ERR_CUDA;
    cudaDeviceProp prop;
    OFB_CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        set_error("device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, prop.major, prop.minor);
        return OFB_ERR_UNSUPPORTED;
    }
    ofb_ctx *c = new (std::nothrow) ofb_ctx();
    if (!c) {
        set_error("out of host memory");
        return OFB_ERR_NOMEM;
    }
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    if (const char *e = getenv("OFB_E2E_LANES")) { // developer overrides for experiments
        const int v = atoi(e);
        if (v >= 1 && v <= OFB_LANES) c->lanes = v;
    }
    if (const char *e = getenv("OFB_E2E_SUB")) c->sub_pairs = atoi(e) > 0 ? atoi(e) : 0;
    if (const char *e = getenv("OFB_HOST_THREADS")) {
        const int v = atoi(e);
        if (v >= 0 && v <= 64) c->host_threads = v;
    }
    e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        set_error("cudaStreamCreate failed: %s", cudaGetErrorString(e));
        delete c;
        return OFB_ERR_CUDA;
    }
    e = cudaEventCreateWithFlags(&c->ws_event, cudaEventDisableTiming);
    if (e != cudaSuccess) {
        set_error("cudaEventCreate failed: %s", cudaGetErrorString(e));
        cudaStreamDestroy(c->stream);
        delete c;
        return OFB_ERR_CUDA;
    }
    for (int l = 0; l < OFB_LANES; l++) {
        e = cudaStreamCreateWithFlags(&c->lane_stream[l], cudaStreamNonBlocking);
        if (e != cudaSuccess) {
            set_error("cudaStreamCreate failed: %s", cudaGetErrorString(e));
            delete c;
            return OFB_ERR_CUDA;
        }
    }
    *out = c;
    return OFB_OK;
}

int ofb_ctx_destroy(ofb_ctx *c)
{
    OFB_CHECK_CTX(c);
    {
        DeviceGuard g(c->device);
        if (g.ok) {
            cudaDeviceSynchronize();
            for (auto &r : c->prof) {
                cudaEventDestroy(r.a);
                cudaEventDestroy(r.b);
            }
            if (c->ws) cudaFree(c->ws);
            if (c->bil_lut) cudaFree(c->bil_lut);
            if (c->ws_event) cudaEventDestroy(c->ws_event);
            if (c->stream) cudaStreamDestroy(c->stream);
            for (int l = 0; l < OFB_LANES; l++) {
                if (c->lane_stream[l]) cudaStreamDestroy(c->lane_stream[l]);
                if (c->stage_ev[l]) cudaEventDestroy(c->stage_ev[l]);
            }
            if (c->stage) cudaFreeHost(c->stage);
        }
    }
    delete c->pool;
    delete c;
    return OFB_OK;
}

int ofb_ctx_set_host_threads(ofb_ctx *c, int threads)
{
    OFB_CHECK_CTX(c);
    if (threads < 0 || threads > 64) {
        set_error("host threads %d outside 0..64", threads);
        return OFB_ERR_INVALID;
    }
    if (c->pool && c->pool->threads() != threads) {
        delete c->pool;
        c->pool = nullptr;
    }
    c->host_threads = threads;
    return OFB_OK;
}

int ofb_ctx_get_host_threads(const ofb_ctx *c, int *threads)
{
    OFB_CHECK_CTX(c);
    if (threads) *threads = c->host_threads;
    return OFB_OK;
}

int ofb_c3_extract_host(const unsigned char *src_c3, unsigned char *dst_planar, size_t n_pixels, int threads)
{
    if (!src_c3 || !dst_planar || threads < 1 || threads > 64) {
        set_error("c3_extract_host: bad arguments");
        return OFB_ERR_INVALID;
    }
    try {
        ofb::HostPool pool(threads);
        // (the two-set helper with one set: the second set is empty)
        const size_t half = n_pixels / 2;
        ofb::c3_extract_pair_sets(&pool, src_c3, src_c3 + 3 * half, dst_planar, dst_planar + half, half);
        ofb::c3_extract_channel0(src_c3 + 3 * 2 * half, dst_planar + 2 * half, n_pixels - 2 * half);
    } catch (...) {
        set_error("c3_extract_host: could not start the host threads");
        return OFB_ERR_NOMEM;
    }
    return OFB_OK;
}

int ofb_ctx_device(const ofb_ctx *c, int *device)
{
    OFB_CHECK_CTX(c);
    if (device) *device = c->device;
    return OFB_OK;
}

int ofb_ctx_sm_count(const ofb_ctx *c, int *sm_count)
{
    OFB_CHECK_CTX(c);
    if (sm_count) *sm_count = c->sm_count;
    return OFB_OK;
}

int ofb_ctx_set_solve(ofb_ctx *c, int solve_mode)
{
    OFB_CHECK_CTX(c);
    if (solve_mode != OFB_SOLVE_EXACT && solve_mode != OFB_SOLVE_FAST) {
        set_error("unknown solve mode %d", solve_mode);
        return OFB_ERR_INVALID;
    }
    c->solve_fast = solve_mode == OFB_SOLVE_FAST;
    return OFB_OK;
}

int ofb_ctx_get_solve(const ofb_ctx *c, int *solve_mode)
{
    OFB_CHECK_CTX(c);
    if (solve_mode) *solve_mode = c->solve_fast ? OFB_SOLVE_FAST : OFB_SOLVE_EXACT;
    return OFB_OK;
}

int ofb_ctx_launch_count(const ofb_ctx *c, unsigned long long *count)
{
    OFB_CHECK_CTX(c);
    if (count) *count = c->launches;
    return OFB_OK;
}

int ofb_ctx_profile_enable(ofb_ctx *c, int on)
{
    OFB_CHECK_CTX(c);
    OFB_GUARD(c);
    c->prof_on = on != 0;
    for (auto &r : c->prof) {
        cudaEventDestroy(r.a);
        cudaEventDestroy(r.b);
    }
    c->prof.clear();
    return OFB_OK;
}

int ofb_ctx_profile_read(ofb_ctx *c, int tag, double *ms_sum, unsigned long long *n_records)
{
    OFB_CHECK_CTX(c);
    OFB_GUARD(c);
    double sum = 0.0;
    unsigned long long n = 0;
    for (auto &r : c->prof) {
        if (r.tag != tag) continue;
        OFB_CUDA_TRY(cudaEventSynchronize(r.b));
        float ms = 0.0f;
        OFB_CUDA_TRY(cudaEventElapsedTime(&ms, r.a, r.b));
        sum += ms;
        n++;
    }
    if (ms_sum) *ms_sum = sum;
    if (n_records) *n_records = n;
    return OFB_OK;
}

int ofb_host_alloc(void **ptr, size_t bytes)
{
    if (!ptr) {
        set_error("ptr is NULL");
        return OFB_ERR_INVALID;
    }
    // (write-combined pinned memory for the upload buffers was measured: no difference, 4.58 k Mpx-pairs/s either way)
    cudaError_t e = cudaHostAlloc(ptr, bytes, cudaHostAllocDefault);
    if (e != cudaSuccess) {
        set_error("cudaHostAlloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
        cudaGetLastError();
        return OFB_ERR_NOMEM;
    }
    return OFB_OK;
}

int ofb_host_free(void *ptr)
{
    if (ptr) OFB_CUDA_TRY(cudaFreeHost(ptr));
    return OFB_OK;
}

// ---------------------------------------------------------------------------------------------
// device-resident hot path
// ---------------------------------------------------------------------------------------------
int ofb_flow_pairs_device(ofb_ctx *c, const ofb_params *p, const uint8_t *prev_d, const uint8_t *next_d,
                          size_t pitch_bytes, size_t image_stride_bytes, float *const *flow_levels_d, float *total_flow_d,
                          void *stream)
{
    OFB_CHECK_CTX(c);
    int rc = check_params(p);
    if (rc) return rc;
    if ((rc = check_device_frames(p, prev_d && next_d && flow_levels_d, "NULL frame or flow pointer", pitch_bytes,
                                  image_stride_bytes)))
        return rc;
    for (int k = 0; k < p->levels; k++)
        if (!flow_levels_d[k]) {
            set_error("flow_levels_d[%d] is NULL", k);
            return OFB_ERR_INVALID;
        }
    OFB_GUARD(c);
    Carver cv;
    PairPlan pl;
    plan_pairs(p, &pl, &cv);
    rc = ws_reserve(c, pl.bytes);
    if (rc) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if ((rc = ws_acquire(c, st))) return rc;
    rc = run_pairs_device(c, p, pl, c->ws, prev_d, next_d, pitch_bytes, image_stride_bytes, flow_levels_d, total_flow_d, st);
    if (rc) return rc;
    return ws_release(c, st);
}

int ofb_ctx_reserve_pairs(ofb_ctx *c, const ofb_params *p)
{
    OFB_CHECK_CTX(c);
    int rc = check_params(p);
    if (rc) return rc;
    OFB_GUARD(c);
    Carver cv;
    PairPlan pl;
    plan_pairs(p, &pl, &cv);
    return ws_reserve(c, pl.bytes);
}

int ofb_fb_check_device(ofb_ctx *c, const float *fwd_d, const float *bwd_d, int w, int h, int n_pairs, float flow_scale,
                        float alpha, float beta, uint8_t *status_d, float *err2_d, void *stream)
{
    OFB_CHECK_CTX(c);
    int rc = check_fb_args(flow_scale, alpha, beta);
    if (rc) return rc;
    if ((rc = check_fb_buffers(fwd_d, bwd_d, status_d, err2_d))) return rc;
    OFB_GUARD(c);
    return run_fb_check(c, fwd_d, bwd_d, w, h, n_pairs, flow_scale, alpha, beta, status_d, err2_d, static_cast<cudaStream_t>(stream));
}

int ofb_flow_pairs_fb_device(ofb_ctx *c, const ofb_params *p, const uint8_t *prev_d, const uint8_t *next_d, size_t pitch_bytes,
                             size_t image_stride_bytes, float alpha, float beta, float *fwd_total_d, float *bwd_total_d,
                             uint8_t *status_d, float *err2_d, void *stream)
{
    OFB_CHECK_CTX(c);
    int rc = check_params(p);
    if (rc) return rc;
    if ((rc = check_fb_args(p->flow_scale, alpha, beta))) return rc;
    if ((rc = check_fb_buffers(fwd_total_d, bwd_total_d, status_d, err2_d))) return rc;
    if ((rc = check_device_frames(p, prev_d && next_d, "NULL frame pointer", pitch_bytes, image_stride_bytes))) return rc;
    OFB_GUARD(c);
    PairFbPlan fp;
    plan_pairs_fb(p, &fp);
    rc = ws_reserve(c, fp.bytes);
    if (rc) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if ((rc = ws_acquire(c, st))) return rc;
    if ((rc = run_pairs_fb_device(c, p, fp, c->ws, prev_d, next_d, pitch_bytes, image_stride_bytes, alpha, beta, fwd_total_d,
                                  bwd_total_d, status_d, err2_d, st)))
        return rc;
    return ws_release(c, st);
}

int ofb_ctx_reserve_pairs_fb(ofb_ctx *c, const ofb_params *p)
{
    OFB_CHECK_CTX(c);
    int rc = check_params(p);
    if (rc) return rc;
    OFB_GUARD(c);
    PairFbPlan fp;
    plan_pairs_fb(p, &fp);
    return ws_reserve(c, fp.bytes);
}

int ofb_track_points_device(ofb_ctx *c, const ofb_params *p, const uint8_t *prev_d, const uint8_t *next_d, size_t pitch_bytes,
                            size_t image_stride_bytes, const float *points_d, int n_points, int iters, float eps, float min_eig,
                            float *flow_d, uint8_t *status_d, void *stream)
{
    OFB_CHECK_CTX(c);
    int rc = check_params(p);
    if (rc) return rc;
    if (p->warp_mode != OFB_WARP_BILINEAR) {
        set_error("track_points: warp mode %d (points are sampled bilinearly: OFB_WARP_BILINEAR only)", p->warp_mode);
        return OFB_ERR_INVALID;
    }
    // s256 = flow_scale * 256 must be finite too: rint(d * s256) of an infinite s256 has no integer value
    if (!(std::isfinite(p->flow_scale * 256.0f) && p->flow_scale > 0.0f)) {
        set_error("flow_scale %g must be > 0 with flow_scale * 256 finite", (double)p->flow_scale);
        return OFB_ERR_INVALID;
    }
    if ((rc = check_device_frames(p, prev_d && next_d && points_d && flow_d && status_d, "NULL frame, point, flow or status pointer",
                                  pitch_bytes, image_stride_bytes)))
        return rc;
    if ((reinterpret_cast<uintptr_t>(points_d) | reinterpret_cast<uintptr_t>(flow_d)) & 7) {
        set_error("points and flow must be 8-byte aligned");
        return OFB_ERR_INVALID;
    }
    if (n_points < 1 || n_points > (1 << 24)) {
        set_error("n_points %d outside 1..%d", n_points, 1 << 24);
        return OFB_ERR_INVALID;
    }
    if (iters < 1 || iters > 64) {
        set_error("iters %d outside 1..64", iters);
        return OFB_ERR_INVALID;
    }
    if (!(std::isfinite(eps) && eps >= 0.0f && std::isfinite(min_eig) && min_eig >= 0.0f)) {
        set_error("eps %g / min_eig %g must be finite and >= 0", (double)eps, (double)min_eig);
        return OFB_ERR_INVALID;
    }
    OFB_GUARD(c);
    Carver cv;
    PairPlan pl;
    plan_pairs(p, &pl, &cv);
    rc = ws_reserve(c, pl.bytes);
    if (rc) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if ((rc = ws_acquire(c, st))) return rc;
    PairLevels lv;
    if ((rc = build_pyramids(c, p, pl, c->ws, prev_d, next_d, pitch_bytes, image_stride_bytes, &lv, st))) return rc;
    TrackArgs a = {};
    for (int k = 0; k < p->levels; k++) {
        a.prev[k] = lv.prev[k];
        a.next[k] = lv.next[k];
        a.pitch[k] = lv.pitch[k];
        a.istr[k] = lv.istr[k];
    }
    a.w = p->w;
    a.h = p->h;
    a.levels = p->levels;
    a.n_pairs = p->n_pairs;
    a.n_points = n_points;
    a.points = points_d;
    a.flow = flow_d;
    a.status = status_d;
    a.iters = iters;
    a.eps = eps;
    a.min_eig = min_eig;
    a.flow_scale = p->flow_scale;
    if ((rc = prof_begin(c, OFB_PROFILE_TRACK, st))) return rc;
    if ((rc = launch_track_points(a, p->win, st, &c->launches))) return rc;
    if ((rc = prof_end(c, st))) return rc;
    return ws_release(c, st);
}

// ---- Shi-Tomasi corners: the frame and size limits both entry points share, and the detector's workspace ----------------
static int check_corner_sizes(int w, int h, int n_images, int win)
{
    if (n_images < 1 || n_images > 65535) {
        set_error("corners: n_images %d outside 1..65535", n_images);
        return OFB_ERR_INVALID;
    }
    if (w < 1 || h < 1 || (long long)w * h >= (1ll << 31)) {
        set_error("corners: image %dx%d (w, h >= 1 and w * h < 2^31)", w, h);
        return OFB_ERR_INVALID;
    }
    if (win < 3 || win > OFB_MAX_WINDOW || !(win & 1)) {
        set_error("corners: window %d not supported (odd 3..%d)", win, OFB_MAX_WINDOW);
        return OFB_ERR_UNSUPPORTED;
    }
    return OFB_OK;
}
static int check_corner_frames(const uint8_t *img_d, size_t pitch_bytes, size_t image_stride_bytes, int w, int h, int n_images,
                               int win)
{
    const int rc = check_corner_sizes(w, h, n_images, win);
    if (rc) return rc;
    ofb_params p = {w, h, 1, win, OFB_WARP_BILINEAR, 1.0f, n_images};
    return check_device_frames(&p, img_d != nullptr, "corners: NULL image pointer", pitch_bytes, image_stride_bytes);
}

struct CornerWs {
    CornerPlan cp;
    size_t off_map, off_max, off_beg, off_end, off_kin, off_kout, off_grid, off_sort, sort_bytes, bytes;
};

static int plan_corner_ws(int w, int h, int n, int win, CornerWs *p)
{
    plan_corners(w, h, n, win, &p->cp);
    if (p->cp.total >= (1ll << 31)) {
        set_error("corners: %d images of %dx%d hold %lld candidate slots (the per-image sort takes < 2^31)", n, w, h, p->cp.total);
        return OFB_ERR_UNSUPPORTED;
    }
    int rc = corner_sort_bytes(p->cp.total, n, &p->sort_bytes);
    if (rc) return rc;
    Carver cv;
    p->off_map = cv.take((size_t)w * h * n * sizeof(float));
    p->off_max = cv.take((size_t)n * sizeof(unsigned));
    p->off_beg = cv.take((size_t)n * sizeof(int));
    p->off_end = cv.take((size_t)n * sizeof(int));
    p->off_kin = cv.take((size_t)p->cp.total * 8);
    p->off_kout = cv.take((size_t)p->cp.total * 8);
    p->off_grid = cv.take((size_t)p->cp.iw * p->cp.ih * n * sizeof(int));
    p->off_sort = cv.take(p->sort_bytes);
    p->bytes = cv.off;
    return OFB_OK;
}

int ofb_min_eig_map_device(ofb_ctx *c, const uint8_t *img_d, size_t pitch_bytes, size_t image_stride_bytes, int w, int h,
                           int n_images, int win, float *score_d, void *stream)
{
    OFB_CHECK_CTX(c);
    int rc = check_corner_frames(img_d, pitch_bytes, image_stride_bytes, w, h, n_images, win);
    if (rc) return rc;
    if (!score_d || (reinterpret_cast<uintptr_t>(score_d) & 3)) {
        set_error("corners: score map NULL or not 4-byte aligned");
        return OFB_ERR_INVALID;
    }
    OFB_GUARD(c);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    CornerArgs a = {};
    a.img = img_d;
    a.pitch = pitch_bytes;
    a.istr = image_stride_bytes;
    a.w = w;
    a.h = h;
    a.n = n_images;
    a.m = win / 2 + 1;
    a.map = score_d;
    a.map_stride = (size_t)w * h;
    if ((rc = prof_begin(c, OFB_PROFILE_CORNERS, st))) return rc;
    if ((rc = launch_corner_score(a, win, st, &c->launches))) return rc;
    return prof_end(c, st);
}

int ofb_detect_corners_device(ofb_ctx *c, const uint8_t *img_d, size_t pitch_bytes, size_t image_stride_bytes, int w, int h,
                              int n_images, int win, int max_corners, float quality_level, float min_distance, float min_score,
                              float *corners_d, float *scores_d, int *counts_d, void *stream)
{
    OFB_CHECK_CTX(c);
    int rc = check_corner_frames(img_d, pitch_bytes, image_stride_bytes, w, h, n_images, win);
    if (rc) return rc;
    if (max_corners < 1 || max_corners > (1 << 20)) {
        set_error("corners: max_corners %d outside 1..%d", max_corners, 1 << 20);
        return OFB_ERR_INVALID;
    }
    if (!(std::isfinite(quality_level) && quality_level >= 0.0f && quality_level <= 1.0f)) {
        set_error("corners: quality_level %g must be finite and in [0, 1]", (double)quality_level);
        return OFB_ERR_INVALID;
    }
    if (!(std::isfinite(min_distance) && min_distance >= 0.0f && std::isfinite(min_score) && min_score >= 0.0f)) {
        set_error("corners: min_distance %g / min_score %g must be finite and >= 0", (double)min_distance, (double)min_score);
        return OFB_ERR_INVALID;
    }
    if (!corners_d || !counts_d) {
        set_error("corners: NULL corner or count pointer");
        return OFB_ERR_INVALID;
    }
    if ((reinterpret_cast<uintptr_t>(corners_d) & 7) || (reinterpret_cast<uintptr_t>(scores_d) & 3) ||
        (reinterpret_cast<uintptr_t>(counts_d) & 3)) {
        set_error("corners: corners must be 8-byte aligned, scores and counts 4-byte aligned");
        return OFB_ERR_INVALID;
    }
    OFB_GUARD(c);
    CornerWs ws;
    if ((rc = plan_corner_ws(w, h, n_images, win, &ws))) return rc;
    if ((rc = ws_reserve(c, ws.bytes))) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if ((rc = ws_acquire(c, st))) return rc;
    DetectArgs d = {};
    d.plan = ws.cp;
    d.img = img_d;
    d.pitch = pitch_bytes;
    d.istr = image_stride_bytes;
    d.w = w;
    d.h = h;
    d.n = n_images;
    d.max_corners = max_corners;
    d.quality_level = quality_level;
    d.min_distance = min_distance;
    d.min_score = min_score;
    d.map = reinterpret_cast<float *>(c->ws + ws.off_map);
    d.max_bits = reinterpret_cast<unsigned *>(c->ws + ws.off_max);
    d.seg_begin = reinterpret_cast<int *>(c->ws + ws.off_beg);
    d.seg_end = reinterpret_cast<int *>(c->ws + ws.off_end);
    d.keys_in = reinterpret_cast<unsigned long long *>(c->ws + ws.off_kin);
    d.keys_out = reinterpret_cast<unsigned long long *>(c->ws + ws.off_kout);
    d.grid = reinterpret_cast<int *>(c->ws + ws.off_grid);
    d.sort_tmp = c->ws + ws.off_sort;
    d.sort_bytes = ws.sort_bytes;
    d.corners = corners_d;
    d.scores = scores_d;
    d.counts = counts_d;
    if ((rc = prof_begin(c, OFB_PROFILE_CORNERS, st))) return rc;
    if ((rc = launch_detect_corners(d, win, st, &c->launches))) return rc;
    if ((rc = prof_end(c, st))) return rc;
    return ws_release(c, st);
}

int ofb_ctx_reserve_corners(ofb_ctx *c, int w, int h, int n_images, int win, int max_corners)
{
    OFB_CHECK_CTX(c);
    int rc = check_corner_sizes(w, h, n_images, win);
    if (rc) return rc;
    if (max_corners < 1 || max_corners > (1 << 20)) {
        set_error("corners: max_corners %d outside 1..%d", max_corners, 1 << 20);
        return OFB_ERR_INVALID;
    }
    OFB_GUARD(c);
    CornerWs ws;
    if ((rc = plan_corner_ws(w, h, n_images, win, &ws))) return rc;
    return ws_reserve(c, ws.bytes);
}

int ofb_pyr_down_device(ofb_ctx *c, const uint8_t *src_d, size_t src_pitch, size_t src_image_stride, int sw, int sh,
                        uint8_t *dst_d, size_t dst_pitch, size_t dst_image_stride, int n_images, void *stream)
{
    OFB_CHECK_CTX(c);
    if (!src_d || !dst_d) {
        set_error("NULL image pointer");
        return OFB_ERR_INVALID;
    }
    OFB_GUARD(c);
    return launch_pyr_down(src_d, src_pitch, src_image_stride, sw, sh, dst_d, dst_pitch, dst_image_stride, n_images, 1,
                           static_cast<cudaStream_t>(stream), &c->launches);
}

int ofb_pyr_down2_device(ofb_ctx *c, const uint8_t *src_d, size_t src_pitch, size_t src_image_stride, int sw, int sh,
                         uint8_t *dst1_d, size_t dst1_pitch, size_t dst1_image_stride, uint8_t *dst2_d, size_t dst2_pitch,
                         size_t dst2_image_stride, int n_images, void *stream)
{
    OFB_CHECK_CTX(c);
    if (!src_d || !dst1_d || !dst2_d) {
        set_error("NULL image pointer");
        return OFB_ERR_INVALID;
    }
    OFB_GUARD(c);
    return launch_pyr_roll(src_d, src_pitch, src_image_stride, sw, sh, dst1_d, dst1_pitch, dst1_image_stride, dst2_d, dst2_pitch,
                           dst2_image_stride, n_images, static_cast<cudaStream_t>(stream), &c->launches, nullptr, nullptr, nullptr,
                           c->sm_count);
}

int ofb_pyr_down_strip_device(ofb_ctx *c, const uint8_t *src_d, size_t src_pitch, int sw, int src_rows, int src_y_off,
                              uint8_t *dst_d, size_t dst_pitch, int dst_y0, int dst_y1, void *stream)
{
    OFB_CHECK_CTX(c);
    if (!src_d || !dst_d) {
        set_error("NULL image pointer");
        return OFB_ERR_INVALID;
    }
    OFB_GUARD(c);
    return launch_pyr_down_strip(src_d, src_pitch, sw, src_rows, src_y_off, dst_d, dst_pitch, dst_y0, dst_y1,
                                 static_cast<cudaStream_t>(stream), &c->launches);
}

int ofb_lk_level_device(ofb_ctx *c, const uint8_t *prev_d, const uint8_t *next_d, size_t pitch_bytes,
                        size_t image_stride_bytes, int w, int h, int n_pairs, int win, int warp_mode, float flow_scale,
                        const float *cum_in_d, float *flow_out_d, float *cum_out_d, void *stream)
{
    OFB_CHECK_CTX(c);
    if (!prev_d || !next_d || !flow_out_d) {
        set_error("NULL image or flow pointer");
        return OFB_ERR_INVALID;
    }
    OFB_GUARD(c);
    LkLevelArgs a = lk_args_frame(prev_d, next_d, pitch_bytes, image_stride_bytes, w, h, n_pairs, win, warp_mode, flow_scale,
                                  flow_out_d, c->sm_count, c->solve_fast);
    a.cum_in = cum_in_d;
    a.cum_w = w >> 1;
    a.cum_h_global = h >> 1;
    a.cum_y_off = 0;
    a.cum_h_local = h >> 1;
    a.cum_pair_stride = (size_t)(w >> 1) * (h >> 1);
    a.cum_out = cum_out_d;
    if (cum_in_d && ((w >> 1) < 1 || (h >> 1) < 1)) {
        set_error("level %dx%d has no coarser level", w, h);
        return OFB_ERR_INVALID;
    }
    return launch_lk_level(a, static_cast<cudaStream_t>(stream), &c->launches);
}

int ofb_lk_level_strip_device(ofb_ctx *c, const uint8_t *prev_d, const uint8_t *next_d, size_t pitch_bytes, int w,
                              int h_local, int y_off, int h_global, int out_y0, int out_y1, int win, int warp_mode,
                              float flow_scale, const float *cum_in_d, int cum_y_off, int cum_h_local, float *flow_out_d,
                              float *cum_out_d, int *reach_overflow_d, void *stream)
{
    OFB_CHECK_CTX(c);
    if (!prev_d || !next_d || !flow_out_d) {
        set_error("NULL image or flow pointer");
        return OFB_ERR_INVALID;
    }
    if (cum_in_d && warp_mode == OFB_WARP_AS_WRITTEN) {
        set_error("OFB_WARP_AS_WRITTEN needs pixel (0,0) of every coarser level and is not available on row strips");
        return OFB_ERR_UNSUPPORTED;
    }
    if (y_off < 0 || y_off + h_local > h_global) {
        set_error("strip rows [%d,%d) outside the level height %d", y_off, y_off + h_local, h_global);
        return OFB_ERR_INVALID;
    }
    OFB_GUARD(c);
    LkLevelArgs a = lk_args_strip(prev_d, next_d, pitch_bytes, w, h_local, y_off, h_global, out_y0, out_y1, win, warp_mode,
                                  flow_scale, flow_out_d, c->sm_count, c->solve_fast);
    a.cum_in = cum_in_d;
    a.cum_w = w >> 1;
    a.cum_h_global = h_global >> 1;
    a.cum_y_off = cum_y_off;
    a.cum_h_local = cum_h_local;
    a.cum_out = cum_out_d;
    a.reach_overflow = reach_overflow_d;
    return launch_lk_level(a, static_cast<cudaStream_t>(stream), &c->launches);
}

int ofb_c3_to_planar_device(ofb_ctx *c, const uint8_t *src_c3_d, int w, int h, int n_images, uint8_t *dst_d,
                            size_t dst_pitch, size_t dst_image_stride, void *stream)
{
    OFB_CHECK_CTX(c);
    if (!src_c3_d || !dst_d) {
        set_error("NULL image pointer");
        return OFB_ERR_INVALID;
    }
    OFB_GUARD(c);
    return launch_c3_to_planar(src_c3_d, w, h, n_images, dst_d, dst_pitch, dst_image_stride,
                               static_cast<cudaStream_t>(stream), &c->launches);
}

// ---------------------------------------------------------------------------------------------
// host-pointer entry points (synchronous)
// ---------------------------------------------------------------------------------------------
int ofb_gauss_pyramid_host_u8c3(ofb_ctx *c, unsigned char **pyramid, int w, int h, int levels)
{
    OFB_CHECK_CTX(c);
    if (!pyramid || levels < 1 || levels > OFB_MAX_LEVELS || w < 1 || h < 1 || (w >> (levels - 1)) < 1 ||
        (h >> (levels - 1)) < 1) {
        set_error("gauss_pyramid: bad arguments (w %d h %d levels %d)", w, h, levels);
        return OFB_ERR_INVALID;
    }
    for (int k = 0; k < levels; k++)
        if (!pyramid[k]) {
            set_error("gauss_pyramid: pyramid[%d] is NULL", k);
            return OFB_ERR_INVALID;
        }
    if (levels == 1) return OFB_OK;
    OFB_GUARD(c);
    Carver cv;
    size_t off[OFB_MAX_LEVELS];
    for (int k = 0; k < levels; k++) off[k] = cv.take((size_t)(w >> k) * (h >> k) * 3);
    int rc = ws_reserve(c, cv.off);
    if (rc) return rc;
    cudaStream_t st = c->stream;
    if ((rc = ws_acquire(c, st))) return rc;
    OFB_CUDA_TRY(cudaMemcpyAsync(c->ws + off[0], pyramid[0], (size_t)w * h * 3, cudaMemcpyHostToDevice, st));
    for (int k = 1; k < levels; k++) {
        const int sw = w >> (k - 1), sh = h >> (k - 1), dw = w >> k, dh = h >> k;
        rc = launch_pyr_down(c->ws + off[k - 1], (size_t)sw * 3, 0, sw, sh, c->ws + off[k], (size_t)dw * 3, 0, 1, 3, st,
                             &c->launches);
        if (rc) return rc;
        OFB_CUDA_TRY(cudaMemcpyAsync(pyramid[k], c->ws + off[k], (size_t)dw * dh * 3, cudaMemcpyDeviceToHost, st));
    }
    OFB_CUDA_TRY(cudaStreamSynchronize(st));
    return OFB_OK;
}

int ofb_calc_opt_flow_host_u8c3(ofb_ctx *c, const unsigned char *prev, const unsigned char *next, int w, int h,
                                float **optFlowPyramid, int level, int maxLevel, int win, int warp_mode, float flow_scale)
{
    OFB_CHECK_CTX(c);
    if (!prev || !next || !optFlowPyramid || w < 1 || h < 1 || level < 0 || level >= maxLevel ||
        maxLevel > OFB_MAX_LEVELS) {
        set_error("calc_opt_flow: bad arguments (w %d h %d level %d maxLevel %d)", w, h, level, maxLevel);
        return OFB_ERR_INVALID;
    }
    for (int k = level; k < maxLevel; k++) {
        if (!optFlowPyramid[k]) {
            set_error("calc_opt_flow: optFlowPyramid[%d] is NULL", k);
            return OFB_ERR_INVALID;
        }
        if ((w >> (k - level)) < 1 || (h >> (k - level)) < 1) {
            set_error("calc_opt_flow: level %d of a %dx%d level-%d image is empty", k, w, h, level);
            return OFB_ERR_INVALID;
        }
    }
    OFB_GUARD(c);
    const size_t pitch = align_up((size_t)w, 64);
    Carver cv;
    const size_t off_c3 = cv.take((size_t)w * h * 3 * 2);
    const size_t off_p = cv.take(pitch * h), off_n = cv.take(pitch * h);
    const size_t off_flow = cv.take((size_t)w * h * 8);
    size_t off_res[OFB_MAX_LEVELS], off_cum[OFB_MAX_LEVELS];
    for (int k = level + 1; k < maxLevel; k++) {
        const size_t n = (size_t)(w >> (k - level)) * (h >> (k - level));
        off_res[k] = cv.take(n * 8);
        off_cum[k] = cv.take(n * 8);
    }
    int rc = ws_reserve(c, cv.off);
    if (rc) return rc;
    cudaStream_t st = c->stream;
    if ((rc = ws_acquire(c, st))) return rc;
    uint8_t *B = c->ws;
    const size_t c3 = (size_t)w * h * 3;
    OFB_CUDA_TRY(cudaMemcpyAsync(B + off_c3, prev, c3, cudaMemcpyHostToDevice, st));
    OFB_CUDA_TRY(cudaMemcpyAsync(B + off_c3 + c3, next, c3, cudaMemcpyHostToDevice, st));
    rc = launch_c3_to_planar(B + off_c3, w, h, 1, B + off_p, pitch, pitch * h, st, &c->launches);
    if (rc) return rc;
    rc = launch_c3_to_planar(B + off_c3 + c3, w, h, 1, B + off_n, pitch, pitch * h, st, &c->launches);
    if (rc) return rc;
    // cumulative flow of level+1 from the residual flows the caller holds (main.cu:136-147)
    const float *cum_in = nullptr;
    for (int k = maxLevel - 1; k > level; k--) {
        const int wk = w >> (k - level), hk = h >> (k - level);
        OFB_CUDA_TRY(cudaMemcpyAsync(B + off_res[k], optFlowPyramid[k], (size_t)wk * hk * 8, cudaMemcpyHostToDevice, st));
        if (k == maxLevel - 1) {
            cum_in = reinterpret_cast<const float *>(B + off_res[k]);
        } else {
            rc = launch_compose_cum(reinterpret_cast<const float *>(B + off_res[k]), cum_in, wk, hk, 1,
                                    reinterpret_cast<float *>(B + off_cum[k]), st, &c->launches);
            if (rc) return rc;
            cum_in = reinterpret_cast<const float *>(B + off_cum[k]);
        }
    }
    LkLevelArgs a = lk_args_frame(B + off_p, B + off_n, pitch, pitch * h, w, h, 1, win, warp_mode, flow_scale,
                                  reinterpret_cast<float *>(B + off_flow), c->sm_count, c->solve_fast);
    a.cum_in = cum_in;
    a.cum_w = w >> 1;
    a.cum_h_global = h >> 1;
    a.cum_h_local = h >> 1;
    rc = launch_lk_level(a, st, &c->launches);
    if (rc) return rc;
    OFB_CUDA_TRY(cudaMemcpyAsync(optFlowPyramid[level], B + off_flow, (size_t)w * h * 8, cudaMemcpyDeviceToHost, st));
    OFB_CUDA_TRY(cudaStreamSynchronize(st));
    return OFB_OK;
}

int ofb_conv_3ch_1ch_u8_f32_host(ofb_ctx *c, const unsigned char *src_h, int w, int h, float *dest_h, const float *mask,
                                 int mw, int mh)
{
    OFB_CHECK_CTX(c);
    if (!src_h || !dest_h || !mask || w < 1 || h < 1) {
        set_error("conv: bad arguments");
        return OFB_ERR_INVALID;
    }
    OFB_GUARD(c);
    Carver cv;
    const size_t off_s = cv.take((size_t)w * h * 3), off_d = cv.take((size_t)w * h * 4);
    int rc = ws_reserve(c, cv.off);
    if (rc) return rc;
    cudaStream_t st = c->stream;
    if ((rc = ws_acquire(c, st))) return rc;
    OFB_CUDA_TRY(cudaMemcpyAsync(c->ws + off_s, src_h, (size_t)w * h * 3, cudaMemcpyHostToDevice, st));
    rc = launch_conv_c3_f32(c->ws + off_s, w, h, reinterpret_cast<float *>(c->ws + off_d), mask, mw, mh, st, &c->launches);
    if (rc) return rc;
    OFB_CUDA_TRY(cudaMemcpyAsync(dest_h, c->ws + off_d, (size_t)w * h * 4, cudaMemcpyDeviceToHost, st));
    OFB_CUDA_TRY(cudaStreamSynchronize(st));
    return OFB_OK;
}

int ofb_srm_1ch_f32_host(ofb_ctx *c, const float *arr1_h, const float *arr2_h, int w, int h, int ww, int wh,
                         float *dest_h)
{
    OFB_CHECK_CTX(c);
    if (!arr1_h || !arr2_h || !dest_h || w < 1 || h < 1) {
        set_error("srm: bad arguments");
        return OFB_ERR_INVALID;
    }
    OFB_GUARD(c);
    const size_t n = (size_t)w * h * 4;
    Carver cv;
    const size_t oa = cv.take(n), ob = cv.take(n), od = cv.take(n);
    int rc = ws_reserve(c, cv.off);
    if (rc) return rc;
    cudaStream_t st = c->stream;
    if ((rc = ws_acquire(c, st))) return rc;
    OFB_CUDA_TRY(cudaMemcpyAsync(c->ws + oa, arr1_h, n, cudaMemcpyHostToDevice, st));
    const float *bdev = reinterpret_cast<const float *>(c->ws + oa);
    if (arr2_h != arr1_h) {
        OFB_CUDA_TRY(cudaMemcpyAsync(c->ws + ob, arr2_h, n, cudaMemcpyHostToDevice, st));
        bdev = reinterpret_cast<const float *>(c->ws + ob);
    }
    rc = launch_srm_f32(reinterpret_cast<const float *>(c->ws + oa), bdev, w, h, ww, wh,
                        reinterpret_cast<float *>(c->ws + od), st, &c->launches);
    if (rc) return rc;
    OFB_CUDA_TRY(cudaMemcpyAsync(dest_h, c->ws + od, n, cudaMemcpyDeviceToHost, st));
    OFB_CUDA_TRY(cudaStreamSynchronize(st));
    return OFB_OK;
}

int ofb_inverse_matrix_f32_host(ofb_ctx *c, const float *sumIx2, const float *sumIy2, const float *sumIxIy,
                                const float *sumIxIt, const float *sumIyIt, float **optFlowPyramid, int level, int w, int h)
{
    OFB_CHECK_CTX(c);
    if (!sumIx2 || !sumIy2 || !sumIxIy || !sumIxIt || !sumIyIt || !optFlowPyramid || level < 0 || !optFlowPyramid[level] ||
        w < 1 || h < 1) {
        set_error("inverse_matrix: bad arguments");
        return OFB_ERR_INVALID;
    }
    OFB_GUARD(c);
    const size_t n = (size_t)w * h * 4;
    Carver cv;
    size_t o[5];
    for (int k = 0; k < 5; k++) o[k] = cv.take(n);
    const size_t of = cv.take(2 * n);
    int rc = ws_reserve(c, cv.off);
    if (rc) return rc;
    cudaStream_t st = c->stream;
    if ((rc = ws_acquire(c, st))) return rc;
    const float *src[5] = {sumIx2, sumIy2, sumIxIy, sumIxIt, sumIyIt};
    for (int k = 0; k < 5; k++) OFB_CUDA_TRY(cudaMemcpyAsync(c->ws + o[k], src[k], n, cudaMemcpyHostToDevice, st));
    rc = launch_inverse_f32(reinterpret_cast<const float *>(c->ws + o[0]), reinterpret_cast<const float *>(c->ws + o[1]),
                            reinterpret_cast<const float *>(c->ws + o[2]), reinterpret_cast<const float *>(c->ws + o[3]),
                            reinterpret_cast<const float *>(c->ws + o[4]), reinterpret_cast<float *>(c->ws + of), w * h,
                            st, &c->launches);
    if (rc) return rc;
    OFB_CUDA_TRY(cudaMemcpyAsync(optFlowPyramid[level], c->ws + of, 2 * n, cudaMemcpyDeviceToHost, st));
    OFB_CUDA_TRY(cudaStreamSynchronize(st));
    return OFB_OK;
}

// flow_levels_h: NULL, or an array whose NULL entries are levels the caller does not want downloaded; total_flow_h: NULL
// or the level-0 composition (main.cu:136-147).  At least one output.
static int flow_pairs_host_impl(ofb_ctx *c, const ofb_params *p, const unsigned char *prev_h, const unsigned char *next_h,
                                int channels, float *const *flow_levels_h, float *total_flow_h)
{
    OFB_CHECK_CTX(c);
    int rc = check_params(p);
    if (rc) return rc;
    if (!prev_h || !next_h || (!flow_levels_h && !total_flow_h) || (channels != 1 && channels != 3)) {
        set_error("flow_pairs_host: bad arguments (channels %d)", channels);
        return OFB_ERR_INVALID;
    }
    OFB_GUARD(c);
    size_t off_flow[OFB_MAX_LEVELS], off_total = 0, plan_base = 0;
    PairPlan pl;
    auto plan_lane = [&](int sub, Carver *cv) {
        for (int k = 0; k < p->levels; k++) off_flow[k] = cv->take((size_t)(p->w >> k) * (p->h >> k) * 8 * sub);
        if (total_flow_h) off_total = cv->take((size_t)p->w * p->h * 8 * sub);
        plan_base = cv->off;
        ofb_params ps = *p;
        ps.n_pairs = sub;
        Carver cv2;
        plan_pairs(&ps, &pl, &cv2);
        return plan_base + pl.bytes;
    };
    auto run_sub = [&](const HostSub &s) -> int {
        const int cnt = s.p.n_pairs;
        float *flow_d[OFB_MAX_LEVELS];
        for (int k = 0; k < p->levels; k++) flow_d[k] = reinterpret_cast<float *>(s.B + off_flow[k]);
        float *total_d = total_flow_h ? reinterpret_cast<float *>(s.B + off_total) : nullptr;
        // (one level: the total flow is the residual flow, the kernel has nothing to compose)
        int rc = run_pairs_device(c, &s.p, pl, s.B + plan_base, s.prev0, s.next0, s.pitch0, s.istride0, flow_d,
                                  p->levels > 1 ? total_d : nullptr, s.st);
        if (rc) return rc;
        for (int k = p->levels - 1; k >= 0; k--) {
            if (!flow_levels_h || !flow_levels_h[k]) continue;
            const size_t per_pair = (size_t)(p->w >> k) * (p->h >> k) * 2; // floats
            OFB_CUDA_TRY(cudaMemcpyAsync(flow_levels_h[k] + per_pair * s.first, flow_d[k], per_pair * 4 * cnt,
                                         cudaMemcpyDeviceToHost, s.st));
        }
        if (total_flow_h) {
            const size_t per_pair = (size_t)p->w * p->h * 2;
            OFB_CUDA_TRY(cudaMemcpyAsync(total_flow_h + per_pair * s.first, p->levels > 1 ? total_d : flow_d[0], per_pair * 4 * cnt,
                                         cudaMemcpyDeviceToHost, s.st));
        }
        return OFB_OK;
    };
    return host_pipeline(c, p, prev_h, next_h, channels, plan_lane, run_sub);
}

int ofb_flow_pairs_host(ofb_ctx *c, const ofb_params *p, const unsigned char *prev_h, const unsigned char *next_h,
                        int channels, float *const *flow_levels_h)
{
    if (!flow_levels_h) {
        set_error("flow_pairs_host: flow_levels_h is NULL");
        return OFB_ERR_INVALID;
    }
    if (p)
        for (int k = 0; k < p->levels && k < OFB_MAX_LEVELS; k++)
            if (!flow_levels_h[k]) {
                set_error("flow_levels_h[%d] is NULL", k);
                return OFB_ERR_INVALID;
            }
    return flow_pairs_host_impl(c, p, prev_h, next_h, channels, flow_levels_h, nullptr);
}

int ofb_flow_pairs_host_ex(ofb_ctx *c, const ofb_params *p, const unsigned char *prev_h, const unsigned char *next_h,
                           int channels, float *const *flow_levels_h, float *total_flow_h)
{
    return flow_pairs_host_impl(c, p, prev_h, next_h, channels, flow_levels_h, total_flow_h);
}

int ofb_flow_pairs_fb_host(ofb_ctx *c, const ofb_params *p, const unsigned char *prev_h, const unsigned char *next_h, int channels,
                           float alpha, float beta, float *fwd_total_h, float *bwd_total_h, uint8_t *status_h, float *err2_h)
{
    OFB_CHECK_CTX(c);
    int rc = check_params(p);
    if (rc) return rc;
    if ((rc = check_fb_args(p->flow_scale, alpha, beta))) return rc;
    if (!prev_h || !next_h || !fwd_total_h || !status_h || (channels != 1 && channels != 3)) {
        set_error("flow_pairs_fb_host: bad arguments (NULL frame, fwd_total_h or status_h, or channels %d)", channels);
        return OFB_ERR_INVALID;
    }
    OFB_GUARD(c);
    // a lane: both totals, status and err2 of a sub-batch, then the workspace of ofb_flow_pairs_fb_device
    size_t off_fwd = 0, off_bwd = 0, off_status = 0, off_err2 = 0, plan_base = 0;
    PairFbPlan fp;
    auto plan_lane = [&](int sub, Carver *cv) {
        const size_t px = (size_t)p->w * p->h * sub;
        off_fwd = cv->take(px * 8);
        off_bwd = cv->take(px * 8);
        off_status = cv->take(px);
        if (err2_h) off_err2 = cv->take(px * 4);
        plan_base = cv->off;
        ofb_params ps = *p;
        ps.n_pairs = sub;
        plan_pairs_fb(&ps, &fp);
        return plan_base + fp.bytes;
    };
    auto run_sub = [&](const HostSub &s) -> int {
        float *fwd = reinterpret_cast<float *>(s.B + off_fwd), *bwd = reinterpret_cast<float *>(s.B + off_bwd);
        uint8_t *status = s.B + off_status;
        float *err2 = err2_h ? reinterpret_cast<float *>(s.B + off_err2) : nullptr;
        int rc = run_pairs_fb_device(c, &s.p, fp, s.B + plan_base, s.prev0, s.next0, s.pitch0, s.istride0, alpha, beta, fwd, bwd,
                                     status, err2, s.st);
        if (rc) return rc;
        const size_t px = (size_t)p->w * p->h, at = px * s.first, cnt = s.p.n_pairs;
        OFB_CUDA_TRY(cudaMemcpyAsync(fwd_total_h + 2 * at, fwd, px * 8 * cnt, cudaMemcpyDeviceToHost, s.st));
        if (bwd_total_h) OFB_CUDA_TRY(cudaMemcpyAsync(bwd_total_h + 2 * at, bwd, px * 8 * cnt, cudaMemcpyDeviceToHost, s.st));
        OFB_CUDA_TRY(cudaMemcpyAsync(status_h + at, status, px * cnt, cudaMemcpyDeviceToHost, s.st));
        if (err2_h) OFB_CUDA_TRY(cudaMemcpyAsync(err2_h + at, err2, px * 4 * cnt, cudaMemcpyDeviceToHost, s.st));
        return OFB_OK;
    };
    return host_pipeline(c, p, prev_h, next_h, channels, plan_lane, run_sub);
}

// ---------------------------------------------------------------------------------------------
// pre-processing and the frame loop
// ---------------------------------------------------------------------------------------------
int ofb_grayscale_avg_host_u8c3(ofb_ctx *c, const unsigned char *src_h, unsigned char *dest_h, int h, int w)
{
    OFB_CHECK_CTX(c);
    if (!src_h || !dest_h || w < 1 || h < 1) {
        set_error("grayscale_avg: bad arguments");
        return OFB_ERR_INVALID;
    }
    OFB_GUARD(c);
    const size_t n = (size_t)w * h * 3;
    Carver cv;
    const size_t os = cv.take(n), od = cv.take(n);
    int rc = ws_reserve(c, cv.off);
    if (rc) return rc;
    cudaStream_t st = c->stream;
    if ((rc = ws_acquire(c, st))) return rc;
    OFB_CUDA_TRY(cudaMemcpyAsync(c->ws + os, src_h, n, cudaMemcpyHostToDevice, st));
    rc = launch_grayscale(c->ws + os, w, h, c->ws + od, nullptr, 0, st, &c->launches);
    if (rc) return rc;
    OFB_CUDA_TRY(cudaMemcpyAsync(dest_h, c->ws + od, n, cudaMemcpyDeviceToHost, st));
    OFB_CUDA_TRY(cudaStreamSynchronize(st));
    return OFB_OK;
}

int ofb_bilinear_filter_host_u8c3(ofb_ctx *c, const unsigned char *src, const unsigned char *gray, unsigned char *dest,
                                  int w, int h, int ww, int wh, double sigmaS, double sigmaB)
{
    OFB_CHECK_CTX(c);
    if (!src || !gray || !dest || w < 1 || h < 1) {
        set_error("bilinear_filter: bad arguments");
        return OFB_ERR_INVALID;
    }
    OFB_GUARD(c);
    const size_t n = (size_t)w * h * 3;
    Carver cv;
    const size_t os = cv.take(n), og = cv.take(n), od = cv.take(n), ol = cv.take(256 * sizeof(double));
    int rc = ws_reserve(c, cv.off);
    if (rc) return rc;
    cudaStream_t st = c->stream;
    if ((rc = ws_acquire(c, st))) return rc;
    OFB_CUDA_TRY(cudaMemcpyAsync(c->ws + os, src, n, cudaMemcpyHostToDevice, st));
    const uint8_t *gd = c->ws + os;
    if (gray != src) {
        OFB_CUDA_TRY(cudaMemcpyAsync(c->ws + og, gray, n, cudaMemcpyHostToDevice, st));
        gd = c->ws + og;
    }
    rc = launch_bilateral(c->ws + os, gd, (size_t)w * 3, 3, w, h, ww, wh, sigmaS, sigmaB,
                          reinterpret_cast<double *>(c->ws + ol), c->ws + od, (size_t)w * 3, st, &c->launches);
    if (rc) return rc;
    OFB_CUDA_TRY(cudaMemcpyAsync(dest, c->ws + od, n, cudaMemcpyDeviceToHost, st));
    OFB_CUDA_TRY(cudaStreamSynchronize(st));
    return OFB_OK;
}

int ofb_bilateral_planar_device(ofb_ctx *c, const uint8_t *gray_d, size_t pitch, int w, int h, int ww, int wh, double sigmaS,
                                double sigmaB, uint8_t *dst_d, size_t dst_pitch, void *stream)
{
    OFB_CHECK_CTX(c);
    if (!gray_d || !dst_d) {
        set_error("NULL image pointer");
        return OFB_ERR_INVALID;
    }
    OFB_GUARD(c);
    if (!c->bil_lut) OFB_CUDA_TRY(cudaMalloc(reinterpret_cast<void **>(&c->bil_lut), 256 * sizeof(double)));
    return launch_bilateral(gray_d, gray_d, pitch, 1, w, h, ww, wh, sigmaS, sigmaB, c->bil_lut, dst_d, dst_pitch,
                            static_cast<cudaStream_t>(stream), &c->launches);
}

// ---- SURVEY 8f row 4: debug derivative views (main.cu:19-92) -----------------------------------------------------

int ofb_conv_3ch_1ch_u8_u8_host(ofb_ctx *c, const unsigned char *src_h, int w, int h, unsigned char *dest_h, const float *mask,
                                int mw, int mh)
{
    OFB_CHECK_CTX(c);
    if (!src_h || !dest_h || !mask || w < 1 || h < 1) {
        set_error("conv (u8): bad arguments");
        return OFB_ERR_INVALID;
    }
    OFB_GUARD(c);
    const size_t n = (size_t)w * h;
    Carver cv;
    const size_t os = cv.take(n * 3), od = cv.take(n);
    int rc = ws_reserve(c, cv.off);
    if (rc) return rc;
    cudaStream_t st = c->stream;
    if ((rc = ws_acquire(c, st))) return rc;
    OFB_CUDA_TRY(cudaMemcpyAsync(c->ws + os, src_h, n * 3, cudaMemcpyHostToDevice, st));
    rc = launch_conv_c3_u8(c->ws + os, w, h, c->ws + od, mask, mw, mh, st, &c->launches);
    if (rc) return rc;
    OFB_CUDA_TRY(cudaMemcpyAsync(dest_h, c->ws + od, n, cudaMemcpyDeviceToHost, st));
    OFB_CUDA_TRY(cudaStreamSynchronize(st));
    return OFB_OK;
}

int ofb_debug_view_host_u8c3(ofb_ctx *c, const unsigned char *prev_level_h, const unsigned char *cur_level_h, int w, int h,
                             int level, int which, unsigned char *out_h)
{
    OFB_CHECK_CTX(c);
    if (!cur_level_h || !out_h || (which == OFB_VIEW_T && !prev_level_h) || w < 1 || h < 1 || level < 0 || level > 12) {
        set_error("debug_view: bad arguments");
        return OFB_ERR_INVALID;
    }
    OFB_GUARD(c);
    const size_t n = (size_t)w * h, no = ((size_t)w << level) * ((size_t)h << level);
    Carver cv;
    const size_t oc = cv.take(n * 3), op = cv.take(n * 3), oo = cv.take(no);
    int rc = ws_reserve(c, cv.off);
    if (rc) return rc;
    cudaStream_t st = c->stream;
    if ((rc = ws_acquire(c, st))) return rc;
    OFB_CUDA_TRY(cudaMemcpyAsync(c->ws + oc, cur_level_h, n * 3, cudaMemcpyHostToDevice, st));
    if (which == OFB_VIEW_T) OFB_CUDA_TRY(cudaMemcpyAsync(c->ws + op, prev_level_h, n * 3, cudaMemcpyHostToDevice, st));
    rc = launch_debug_view(c->ws + op, c->ws + oc, w, h, level, which, c->ws + oo, st, &c->launches);
    if (rc) return rc;
    OFB_CUDA_TRY(cudaMemcpyAsync(out_h, c->ws + oo, no, cudaMemcpyDeviceToHost, st));
    OFB_CUDA_TRY(cudaStreamSynchronize(st));
    return OFB_OK;
}

// ---- SURVEY 8f row 3: flow composition and export (the headless part of main.cu:114-174) ----------------------

int ofb_compose_flow_host(ofb_ctx *c, float *const *flow_pyramid_h, int w, int h, int levels, int level, float *total_h)
{
    OFB_CHECK_CTX(c);
    if (!flow_pyramid_h || !total_h || w < 1 || h < 1 || levels < 1 || levels > OFB_MAX_LEVELS || level < 0 || level >= levels ||
        (w >> (levels - 1)) < 1 || (h >> (levels - 1)) < 1) {
        set_error("compose_flow: bad arguments (w %d h %d levels %d level %d)", w, h, levels, level);
        return OFB_ERR_INVALID;
    }
    for (int k = level; k < levels; k++)
        if (!flow_pyramid_h[k]) {
            set_error("compose_flow: flow_pyramid[%d] is NULL", k);
            return OFB_ERR_INVALID;
        }
    OFB_GUARD(c);
    // device: residual flow of levels level..levels-1 and two ping-pong cumulative buffers of the finest size
    Carver cv;
    size_t off_res[OFB_MAX_LEVELS];
    for (int k = level; k < levels; k++) off_res[k] = cv.take((size_t)(w >> k) * (h >> k) * 8);
    const size_t n0 = (size_t)(w >> level) * (h >> level) * 8;
    const size_t off_a = cv.take(n0), off_b = cv.take(n0);
    int rc = ws_reserve(c, cv.off);
    if (rc) return rc;
    cudaStream_t st = c->stream;
    if ((rc = ws_acquire(c, st))) return rc;
    for (int k = level; k < levels; k++)
        OFB_CUDA_TRY(cudaMemcpyAsync(c->ws + off_res[k], flow_pyramid_h[k], (size_t)(w >> k) * (h >> k) * 8,
                                     cudaMemcpyHostToDevice, st));
    // coarse to fine: cum_{L-1} = flow_{L-1}; cum_k = 2*cum_{k+1}[i>>1][j>>1] + flow_k
    const float *cum = nullptr;
    size_t cur = off_a, other = off_b;
    for (int k = levels - 1; k >= level; k--) {
        rc = launch_compose_cum(reinterpret_cast<const float *>(c->ws + off_res[k]), cum, w >> k, h >> k, 1,
                                reinterpret_cast<float *>(c->ws + cur), st, &c->launches);
        if (rc) return rc;
        cum = reinterpret_cast<const float *>(c->ws + cur);
        std::swap(cur, other);
    }
    OFB_CUDA_TRY(cudaMemcpyAsync(total_h, cum, n0, cudaMemcpyDeviceToHost, st));
    OFB_CUDA_TRY(cudaStreamSynchronize(st));
    return OFB_OK;
}

int ofb_flow_arrows_host(ofb_ctx *c, float *const *flow_pyramid_h, int w, int h, int levels, int level, int arrow_res,
                         int *arrows_xyxy, int max_arrows, int *n_arrows)
{
    OFB_CHECK_CTX(c);
    if (!n_arrows || arrow_res < 1 || max_arrows < 0 || (max_arrows > 0 && !arrows_xyxy)) {
        set_error("flow_arrows: bad arguments");
        return OFB_ERR_INVALID;
    }
    if (level < 0 || level >= levels || w < 1 || h < 1) {
        set_error("flow_arrows: bad geometry (w %d h %d levels %d level %d)", w, h, levels, level);
        return OFB_ERR_INVALID;
    }
    const int wl = w >> level, hl = h >> level;
    const int step = wl / arrow_res; // main.cu:124
    if (step < 1) {
        set_error("flow_arrows: arrow_res %d exceeds the level width %d", arrow_res, wl);
        return OFB_ERR_INVALID;
    }
    std::vector<float> total((size_t)wl * hl * 2);
    int rc = ofb_compose_flow_host(c, flow_pyramid_h, w, h, levels, level, total.data());
    if (rc) return rc;
    int n = 0;
    for (int i = 0; i < hl; i += step)
        for (int j = 0; j < wl; j += step) {
            float u = total[((size_t)i * wl + j) * 2], v = total[((size_t)i * wl + j) * 2 + 1];
            // main.cu:150-157: clamp to one grid step; NaN compares false and passes through, as in the reference
            if (u > step) u = (float)step;
            else if (u < -step) u = (float)-step;
            if (v > step) v = (float)step;
            else if (v < -step) v = (float)-step;
            // main.cu:159-160 casts float to int; the result is undefined there for NaN (x86 gives INT_MIN, which the
            // sign test then drops): defined here as "no arrow"
            if (u != u || v != v) continue;
            const int ni = (int)(v + (float)i), nj = (int)(u + (float)j);
            if (ni < 0 || nj < 0) continue; // main.cu:163
            if (n < max_arrows) {
                arrows_xyxy[4 * n + 0] = j;
                arrows_xyxy[4 * n + 1] = i;
                arrows_xyxy[4 * n + 2] = nj;
                arrows_xyxy[4 * n + 3] = ni;
            }
            n++;
        }
    *n_arrows = n;
    return OFB_OK;
}

int ofb_write_flo(const char *path, const float *flow_h, int w, int h)
{
    if (!path || !flow_h || w < 1 || h < 1) {
        set_error("write_flo: bad arguments");
        return OFB_ERR_INVALID;
    }
    FILE *f = fopen(path, "wb");
    if (!f) {
        set_error("write_flo: cannot open %s", path);
        return OFB_ERR_INVALID;
    }
    const float tag = 202021.25f; // "PIEH"
    const int32_t dims[2] = {w, h};
    bool ok = fwrite(&tag, 4, 1, f) == 1 && fwrite(dims, 4, 2, f) == 2 &&
              fwrite(flow_h, 8, (size_t)w * h, f) == (size_t)w * h;
    ok = (fclose(f) == 0) && ok;
    if (!ok) {
        set_error("write_flo: short write to %s", path);
        return OFB_ERR_INVALID;
    }
    return OFB_OK;
}

} // extern "C"

// One frame sequence: two device-resident planar pyramids that swap roles every frame (main.cu:270-272).
struct ofb_stream {
    ofb_ctx *ctx = nullptr;
    ofb_params p{};
    int bil_win = 0;
    double sig_s = 0, sig_b = 0;
    int frames = 0;
    uint8_t *mem = nullptr; // all device buffers of the stream in one allocation
    size_t pitch[OFB_MAX_LEVELS] = {}, off_pyr[2][OFB_MAX_LEVELS] = {}, off_bgr = 0, off_gray = 0, off_lut = 0;
    size_t off_flow[OFB_MAX_LEVELS] = {}, off_cum[OFB_MAX_LEVELS] = {}, off_total = 0; // off_cum: levels 1..L-2
    int cur = 0; // which pyramid receives the next frame
    // The forward-backward check (ofb_stream_push_bgr_host_fb), set up by its first call: the backward direction's residual
    // flow, interior cumulative flow and total, status and err2 in one allocation, and a second stream with two events
    // on which the backward level loop runs alongside the forward one.
    uint8_t *fb_mem = nullptr;
    size_t off_bflow[OFB_MAX_LEVELS] = {}, off_bcum[OFB_MAX_LEVELS] = {}, off_btotal = 0, off_status = 0, off_err2 = 0;
    cudaStream_t fb_stream = nullptr;
    cudaEvent_t fb_fork = nullptr, fb_join = nullptr;
};

namespace ofb {

// The stream's two pyramids as a pair: the previous frame's and the current one's.
static PairLevels stream_pair_levels(const ofb_stream *s)
{
    PairLevels lv;
    for (int k = 0; k < s->p.levels; k++) {
        lv.prev[k] = s->mem + s->off_pyr[s->cur ^ 1][k];
        lv.next[k] = s->mem + s->off_pyr[s->cur][k];
        lv.pitch[k] = s->pitch[k];
        lv.istr[k] = s->pitch[k] * (size_t)(s->p.h >> k);
    }
    return lv;
}

// The residual flow of every level and the cumulative flow of levels 1..L-2 of one direction (bwd: in the check's
// allocation).
static void stream_flow(const ofb_stream *s, bool bwd, float **flow, float **cum)
{
    uint8_t *B = bwd ? s->fb_mem : s->mem;
    for (int k = 0; k < s->p.levels; k++) {
        flow[k] = reinterpret_cast<float *>(B + (bwd ? s->off_bflow[k] : s->off_flow[k]));
        cum[k] = k >= 1 && k <= s->p.levels - 2 ? reinterpret_cast<float *>(B + (bwd ? s->off_bcum[k] : s->off_cum[k])) : nullptr;
    }
}

// Upload, grayscale (main.cu:232), bilateral pre-filter (main.cu:240) and pyramid (main.cu:250) of a new frame into the
// stream's current pyramid, on the context stream.
static int stream_new_frame(ofb_stream *s, const unsigned char *frame_bgr)
{
    ofb_ctx *c = s->ctx;
    const ofb_params &p = s->p;
    cudaStream_t st = c->stream;
    uint8_t *B = s->mem;
    const PairLevels lv = stream_pair_levels(s);
    uint8_t *lvl0 = const_cast<uint8_t *>(lv.next[0]);
    OFB_CUDA_TRY(cudaMemcpyAsync(B + s->off_bgr, frame_bgr, (size_t)p.w * p.h * 3, cudaMemcpyHostToDevice, st));
    int rc = launch_grayscale(B + s->off_bgr, p.w, p.h, nullptr, s->bil_win ? B + s->off_gray : lvl0, s->pitch[0], st,
                              &c->launches);
    if (rc) return rc;
    if (s->bil_win) {
        rc = launch_bilateral(B + s->off_gray, B + s->off_gray, s->pitch[0], 1, p.w, p.h, s->bil_win, s->bil_win, s->sig_s,
                              s->sig_b, reinterpret_cast<double *>(B + s->off_lut), lvl0, s->pitch[0], st, &c->launches);
        if (rc) return rc;
    }
    return build_pyramid_levels(c, p.w, p.h, p.levels, lv.next, nullptr, lv.pitch, lv.istr, 1, st);
}

// One push of either kind: the new frame into the current pyramid; from the second frame on, `pair()` enqueues the pair's
// work and downloads.  Once they are done the current pyramid becomes the previous one (main.cu:270-272).
template <class Pair> static int stream_push(ofb_stream *s, const unsigned char *frame_bgr, int *has_flow, Pair pair)
{
    if (has_flow) *has_flow = 0;
    int rc = stream_new_frame(s, frame_bgr);
    if (rc) return rc;
    if (s->frames > 0) {
        if ((rc = pair())) return rc;
        if (has_flow) *has_flow = 1;
    }
    OFB_CUDA_TRY(cudaStreamSynchronize(s->ctx->stream));
    s->cur ^= 1;
    s->frames++;
    return OFB_OK;
}

// The buffers, stream and events of the check (see ofb_stream::fb_mem); nothing once they exist.
static int stream_fb_setup(ofb_stream *s)
{
    if (s->fb_mem) return OFB_OK;
    if (!s->fb_stream) OFB_CUDA_TRY(cudaStreamCreateWithFlags(&s->fb_stream, cudaStreamNonBlocking));
    if (!s->fb_fork) OFB_CUDA_TRY(cudaEventCreateWithFlags(&s->fb_fork, cudaEventDisableTiming));
    if (!s->fb_join) OFB_CUDA_TRY(cudaEventCreateWithFlags(&s->fb_join, cudaEventDisableTiming));
    const ofb_params &p = s->p;
    Carver cv;
    for (int k = 0; k < p.levels; k++) {
        s->off_bflow[k] = cv.take((size_t)(p.w >> k) * (p.h >> k) * 8);
        if (k >= 1 && k <= p.levels - 2) s->off_bcum[k] = cv.take((size_t)(p.w >> k) * (p.h >> k) * 8);
    }
    const size_t px = (size_t)p.w * p.h;
    s->off_btotal = cv.take(px * 8);
    s->off_status = cv.take(px);
    s->off_err2 = cv.take(px * 4);
    cudaError_t e = cudaMalloc(reinterpret_cast<void **>(&s->fb_mem), cv.off);
    if (e != cudaSuccess) {
        s->fb_mem = nullptr;
        set_error("stream forward-backward cudaMalloc(%zu) failed: %s", cv.off, cudaGetErrorString(e));
        cudaGetLastError();
        return OFB_ERR_NOMEM;
    }
    return OFB_OK;
}

// Backward level loop on the stream's second CUDA stream, concurrently with the forward one (OFB_FB_SERIAL=1: after it, on the
// context stream; a developer switch for A/B measurements).
static bool fb_serial()
{
    static const bool on = [] {
        const char *e = getenv("OFB_FB_SERIAL");
        return e && e[0] == '1';
    }();
    return on;
}

// Both directions on the stream's two pyramids, with the level loop of ofb_flow_pairs_fb_device, then the check and the
// downloads, on the context stream.  The two loops read only the pyramids and write disjoint buffers: forked after the
// pyramid and joined before the check, the backward one runs beside the forward one and shortens the chain of one pair's
// small kernels.
static int stream_fb_pair(ofb_stream *s, float alpha, float beta, float *const *flow_levels_h, float *fwd_total_h,
                          float *bwd_total_h, uint8_t *status_h, float *err2_h)
{
    ofb_ctx *c = s->ctx;
    const ofb_params &p = s->p;
    cudaStream_t st = c->stream;
    uint8_t *B = s->mem, *F = s->fb_mem;
    const PairLevels lv = stream_pair_levels(s);
    float *flow[2][OFB_MAX_LEVELS], *cum[2][OFB_MAX_LEVELS];
    stream_flow(s, false, flow[0], cum[0]);
    stream_flow(s, true, flow[1], cum[1]);
    float *fwd = reinterpret_cast<float *>(B + s->off_total), *bwd = reinterpret_cast<float *>(F + s->off_btotal);
    auto backward = [&](cudaStream_t bst) { return run_levels(c, &p, lv, true, flow[1], cum[1], bwd, bst); };
    const bool fork = !fb_serial();
    int rc;
    if (fork) {
        OFB_CUDA_TRY(cudaEventRecord(s->fb_fork, st));
        OFB_CUDA_TRY(cudaStreamWaitEvent(s->fb_stream, s->fb_fork, 0));
        if ((rc = backward(s->fb_stream))) return rc;
        OFB_CUDA_TRY(cudaEventRecord(s->fb_join, s->fb_stream));
    }
    if ((rc = run_levels(c, &p, lv, false, flow[0], cum[0], fwd, st))) return rc;
    if (fork) OFB_CUDA_TRY(cudaStreamWaitEvent(st, s->fb_join, 0));
    else if ((rc = backward(st))) return rc;
    uint8_t *status = F + s->off_status;
    float *err2 = err2_h ? reinterpret_cast<float *>(F + s->off_err2) : nullptr;
    if ((rc = run_fb_check(c, fwd, bwd, p.w, p.h, 1, p.flow_scale, alpha, beta, status, err2, st))) return rc;
    for (int k = p.levels - 1; k >= 0; k--)
        if (flow_levels_h && flow_levels_h[k])
            OFB_CUDA_TRY(cudaMemcpyAsync(flow_levels_h[k], flow[0][k], (size_t)(p.w >> k) * (p.h >> k) * 8, cudaMemcpyDeviceToHost, st));
    const size_t px = (size_t)p.w * p.h;
    OFB_CUDA_TRY(cudaMemcpyAsync(fwd_total_h, fwd, px * 8, cudaMemcpyDeviceToHost, st));
    if (bwd_total_h) OFB_CUDA_TRY(cudaMemcpyAsync(bwd_total_h, bwd, px * 8, cudaMemcpyDeviceToHost, st));
    OFB_CUDA_TRY(cudaMemcpyAsync(status_h, status, px, cudaMemcpyDeviceToHost, st));
    if (err2_h) OFB_CUDA_TRY(cudaMemcpyAsync(err2_h, err2, px * 4, cudaMemcpyDeviceToHost, st));
    return OFB_OK;
}

} // namespace ofb

extern "C" {

int ofb_stream_create(ofb_ctx *c, const ofb_params *p, int bil_win, double bil_sigma_s, double bil_sigma_b, ofb_stream **out)
{
    OFB_CHECK_CTX(c);
    if (!out) {
        set_error("out is NULL");
        return OFB_ERR_INVALID;
    }
    *out = nullptr;
    int rc = check_params(p);
    if (rc) return rc;
    if (p->n_pairs != 1) {
        set_error("a frame sequence solves one pair per frame (n_pairs must be 1)");
        return OFB_ERR_INVALID;
    }
    if (bil_win != 0 && (bil_win < 3 || bil_win > 9 || !(bil_win & 1))) {
        set_error("bilateral window %d not supported (0 = off, or odd 3..9)", bil_win);
        return OFB_ERR_UNSUPPORTED;
    }
    OFB_GUARD(c);
    ofb_stream *s = new (std::nothrow) ofb_stream();
    if (!s) {
        set_error("out of host memory");
        return OFB_ERR_NOMEM;
    }
    s->ctx = c;
    s->p = *p;
    s->bil_win = bil_win;
    s->sig_s = bil_sigma_s;
    s->sig_b = bil_sigma_b;
    Carver cv;
    s->off_bgr = cv.take((size_t)p->w * p->h * 3);
    for (int k = 0; k < p->levels; k++) {
        const int wk = p->w >> k, hk = p->h >> k;
        s->pitch[k] = align_up((size_t)wk, 64);
        s->off_pyr[0][k] = cv.take(s->pitch[k] * hk);
        s->off_pyr[1][k] = cv.take(s->pitch[k] * hk);
        s->off_flow[k] = cv.take((size_t)wk * hk * 8);
        if (k >= 1 && k <= p->levels - 2) s->off_cum[k] = cv.take((size_t)wk * hk * 8);
    }
    s->off_gray = cv.take(s->pitch[0] * p->h);
    s->off_total = cv.take((size_t)p->w * p->h * 8);
    s->off_lut = cv.take(256 * sizeof(double));
    cudaError_t e = cudaMalloc(reinterpret_cast<void **>(&s->mem), cv.off);
    if (e != cudaSuccess) {
        set_error("stream cudaMalloc(%zu) failed: %s", cv.off, cudaGetErrorString(e));
        cudaGetLastError();
        delete s;
        return OFB_ERR_NOMEM;
    }
    e = cudaMemsetAsync(s->mem, 0, cv.off, c->stream);
    if (e != cudaSuccess) {
        set_error("stream cudaMemsetAsync failed: %s", cudaGetErrorString(e));
        cudaGetLastError();
        cudaFree(s->mem);
        delete s;
        return OFB_ERR_CUDA;
    }
    *out = s;
    return OFB_OK;
}

int ofb_stream_destroy(ofb_stream *s)
{
    if (!s) {
        set_error("stream is NULL");
        return OFB_ERR_INVALID;
    }
    {
        DeviceGuard g(s->ctx->device);
        if (g.ok) {
            cudaStreamSynchronize(s->ctx->stream);
            if (s->mem) cudaFree(s->mem);
            if (s->fb_stream) {
                cudaStreamSynchronize(s->fb_stream);
                cudaStreamDestroy(s->fb_stream);
            }
            if (s->fb_mem) cudaFree(s->fb_mem);
            if (s->fb_fork) cudaEventDestroy(s->fb_fork);
            if (s->fb_join) cudaEventDestroy(s->fb_join);
        }
    }
    delete s;
    return OFB_OK;
}

int ofb_stream_push_bgr_host(ofb_stream *s, const unsigned char *frame_bgr, float *const *flow_levels_h, float *total_flow_h,
                             int *has_flow)
{
    if (!s || !frame_bgr) {
        set_error("stream_push: NULL stream or frame");
        return OFB_ERR_INVALID;
    }
    ofb_ctx *c = s->ctx;
    const ofb_params &p = s->p;
    if (s->frames > 0) { // (before anything is enqueued: a rejected call leaves the sequence where it was)
        if (!flow_levels_h) {
            set_error("stream_push: flow_levels_h is NULL");
            return OFB_ERR_INVALID;
        }
        for (int k = 0; k < p.levels; k++)
            if (!flow_levels_h[k]) {
                set_error("stream_push: flow_levels_h[%d] is NULL", k);
                return OFB_ERR_INVALID;
            }
    }
    OFB_GUARD(c);
    return stream_push(s, frame_bgr, has_flow, [&]() -> int {
        cudaStream_t st = c->stream;
        float *flow[OFB_MAX_LEVELS], *cum[OFB_MAX_LEVELS];
        stream_flow(s, false, flow, cum);
        float *total = total_flow_h ? reinterpret_cast<float *>(s->mem + s->off_total) : nullptr;
        int rc = run_levels(c, &p, stream_pair_levels(s), false, flow, cum, total, st);
        if (rc) return rc;
        for (int k = p.levels - 1; k >= 0; k--)
            OFB_CUDA_TRY(cudaMemcpyAsync(flow_levels_h[k], flow[k], (size_t)(p.w >> k) * (p.h >> k) * 8, cudaMemcpyDeviceToHost, st));
        if (total_flow_h) OFB_CUDA_TRY(cudaMemcpyAsync(total_flow_h, total, (size_t)p.w * p.h * 8, cudaMemcpyDeviceToHost, st));
        return OFB_OK;
    });
}

int ofb_stream_push_bgr_host_fb(ofb_stream *s, const unsigned char *frame_bgr, float alpha, float beta, float *const *flow_levels_h,
                                float *fwd_total_h, float *bwd_total_h, uint8_t *status_h, float *err2_h, int *has_flow)
{
    if (!s || !frame_bgr || !fwd_total_h || !status_h) {
        set_error("stream_push_fb: NULL stream, frame, fwd_total_h or status_h");
        return OFB_ERR_INVALID;
    }
    int rc = check_fb_args(s->p.flow_scale, alpha, beta);
    if (rc) return rc;
    OFB_GUARD(s->ctx);
    // (before anything is enqueued: a failed set-up leaves the sequence where it was)
    if ((rc = stream_fb_setup(s))) return rc;
    return stream_push(s, frame_bgr, has_flow, [&]() -> int {
        int rc = stream_fb_pair(s, alpha, beta, flow_levels_h, fwd_total_h, bwd_total_h, status_h, err2_h);
        // (a failure after the fork: the backward loop may still read the pyramid the next push overwrites)
        if (rc) cudaStreamSynchronize(s->fb_stream);
        return rc;
    });
}

} // extern "C"
