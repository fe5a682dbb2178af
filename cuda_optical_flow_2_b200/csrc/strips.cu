// strips.cu -- row-strip solve of ONE large pair over several GPUs (BASELINE configs[4]), native host side.
//
// One process per GPU.  The strip schedule is the one of cuda_optical_flow_2_b200/dist.py (StripPlan: bounds fixed
// on the coarsest level and doubled per finer level, image halo = window radius + stencil + warp reach, coarser
// cumulative-flow halo), but here the whole pair -- own-row upload, per-level halo exchange, pyramid, fused level
// kernels -- is enqueued on one CUDA stream from C++ with no host synchronisation.  Only level-0 image rows are
// exchanged (the coarser levels' halo rows are rebuilt locally), so a pair of L levels costs L exchanges: one for the
// images, L-1 for the cumulative flow.
//
// The halo rows move through peer memory: every rank keeps the buffers its neighbours write into -- the level-0 image
// rows and the coarser cumulative-flow rows -- in ONE device allocation (the arena) whose CUDA IPC handle the
// application all-gathers once.  An exchange is then a store of the SENDER's kernels straight into the receiver's arena
// over NVLink plus an epoch flag raised there, and a wait for that flag on the receiver's stream: no collective, no host
// work beyond at most two launches per exchange.
#include "ofb_common.cuh"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <new>
#include <vector>

struct ofb_ctx; // ofb_api.cu
namespace ofb {
// accessors implemented in ofb_api.cu (ofb_ctx is private to it)
int ctx_device(const ofb_ctx *c);
int ctx_sm_count(const ofb_ctx *c);
int ctx_solve_fast(const ofb_ctx *c);
unsigned long long *ctx_launch_counter(ofb_ctx *c);

// ---- the strip schedule (dist.py: StripPlan) ---------------------------------------------------------------------
struct LevelStrip {
    int w, h;     // size of the whole level
    int y0, y1;   // rows this rank owns (and produces flow for)
    int by0, by1; // rows the level kernel needs: own rows plus halo, clipped to the image
    int cy0, cy1; // rows of the next-coarser level's cumulative flow its buffer holds
    int eb0, eb1; // rows its image buffers hold: [by0, by1) plus what building [eb0, eb1) of the next level takes
};
struct StripPlan {
    int W, H, levels, win, world, reach, r, img_halo;
    int fb_reach = -1; // >= 0: handle of ofb_strips_create_fb (checked pairs); level-0 backward rows beyond the own rows held
    // first row of `rank`'s strip on the coarsest level; coarse_bound(world) is that level's height
    int coarse_bound(int rank) const { return (int)(((long long)rank * (H >> (levels - 1))) / world); }
    // rows [lo, hi) of the level-0 backward total flow that `rank`'s check holds
    void fb_rows(int rank, int *lo, int *hi) const
    {
        const LevelStrip s = level(0, rank);
        *lo = std::max(0, s.y0 - fb_reach);
        *hi = std::min(H, s.y1 + fb_reach + 1);
    }
    LevelStrip level(int k, int rank) const
    {
        const int sh = levels - 1 - k;
        LevelStrip s;
        s.w = W >> k;
        s.h = H >> k;
        s.y0 = coarse_bound(rank) << sh;
        s.y1 = rank == world - 1 ? s.h : coarse_bound(rank + 1) << sh;
        s.by0 = std::max(0, s.y0 - img_halo);
        s.by1 = std::min(s.h, s.y1 + img_halo);
        if (k < levels - 1) {
            const int hc = H >> (k + 1);
            // the kernel looks up cum[(y >> 1)] for the rows it warps (its packed tile: own rows -r-2 .. +r+1)
            s.cy0 = std::max(0, (s.y0 - r - 2) >> 1);
            s.cy1 = std::min(hc, ((s.y1 + r + 1) >> 1) + 1);
        } else {
            s.cy0 = s.cy1 = 0;
        }
        s.eb0 = s.by0;
        s.eb1 = s.by1;
        return s;
    }
    // Every level of one rank.  Only level-0 rows are exchanged; the halo rows of the coarser levels are built
    // locally (each rank repeats a few rows of pyramid work instead of three more exchanges), so a level's buffer
    // also holds the rows 2y-1 .. 2y+1 under every row y of the next level's buffer.
    std::vector<LevelStrip> strips(int rank) const
    {
        std::vector<LevelStrip> v(levels);
        for (int k = levels - 1; k >= 0; k--) {
            v[k] = level(k, rank);
            if (k + 1 < levels) {
                v[k].eb0 = std::min(v[k].by0, std::max(0, 2 * v[k + 1].eb0 - 1));
                v[k].eb1 = std::max(v[k].by1, std::min(v[k].h, 2 * (v[k + 1].eb1 - 1) + 2));
            }
        }
        return v;
    }
};

// ---- peer memory ------------------------------------------------------------------------------------------------
// Arena of one rank: [prev level 0][next level 0][cum_in level 0 .. L-2][flags]; a handle that runs checked pairs also has
// [cum_in_b level 0 .. L-2][fbh: held rows of the backward total flow] before the flags.  Every rank can compute every
// other rank's layout from the plan, so a peer address is (peer arena base) + (offset computed here).
constexpr int PEER_MAX_SEG = 8;   // copy segments per exchange (prev + next rows per destination)
constexpr int PEER_MAX_DST = 4;   // ranks one exchange sends to / receives from
struct ArenaLayout {
    size_t prev0, next0, cum_in[OFB_MAX_LEVELS], cum_in_b[OFB_MAX_LEVELS], fbh, flags, bytes;
    // Exchanges of a pair: 0 = level-0 images, 1 .. L-1 = forward cumulative flow; a checked pair adds L .. 2L-2 = backward
    // cumulative flow and 2L-1 = backward total rows for the check.  nx = L (plain handle) or 2L.
    int world, nx;
    // flags (unsigned): arrive[x * world + src] = epoch of the last exchange x that src completed into this arena;
    //                   done[src] at nx * world + src = last epoch rank src finished reading what this rank pushed;
    //                   counter[x] at (nx + 1) * world + x: blocks of this rank's push kernel that have finished (local);
    //                   pairs at (nx + 1) * world + nx: pairs this rank has completed (local).  The epoch of a pair is
    //                   pairs + 1, read from here by the kernels, so that a captured CUDA graph of one pair replays;
    //                   fused[2 * x + d] after that: CTAs of the level kernel that have pushed their rows of exchange x to
    //                   target d (local; the halo push fused into the level kernels).
    size_t arrive(int x, int src) const { return (size_t)x * world + src; }
    size_t done(int src) const { return (size_t)nx * world + src; }
    size_t counter(int x) const { return (size_t)(nx + 1) * world + x; }
    size_t pairs() const { return (size_t)(nx + 1) * world + nx; }
    size_t fused(int x) const { return pairs() + 1 + 2 * (size_t)x; }
};
static ArenaLayout arena_layout(const StripPlan &pl, int rank)
{
    ArenaLayout a{};
    const std::vector<LevelStrip> v = pl.strips(rank);
    size_t off = 0;
    auto take = [&](size_t n) {
        const size_t o = off;
        off += (n + 255) / 256 * 256;
        return o;
    };
    const size_t pitch0 = ((size_t)v[0].w + 63) / 64 * 64;
    a.prev0 = take(pitch0 * (v[0].eb1 - v[0].eb0));
    a.next0 = take(pitch0 * (v[0].eb1 - v[0].eb0));
    for (int k = 0; k < pl.levels; k++) a.cum_in[k] = take((size_t)(v[k].w >> 1) * std::max(v[k].cy1 - v[k].cy0, 1) * 8);
    a.world = pl.world;
    a.nx = pl.levels;
    if (pl.fb_reach >= 0) {
        for (int k = 0; k < pl.levels; k++) a.cum_in_b[k] = take((size_t)(v[k].w >> 1) * std::max(v[k].cy1 - v[k].cy0, 1) * 8);
        int lo, hi;
        pl.fb_rows(rank, &lo, &hi);
        a.fbh = take((size_t)v[0].w * (hi - lo) * 8);
        a.nx = 2 * pl.levels;
    }
    a.flags = take((a.pairs() + 1 + 2 * (size_t)a.nx) * sizeof(unsigned));
    a.bytes = off;
    return a;
}

// Exchange x of a pair moves rows of one level from the ranks that own them into the window of that level other ranks'
// buffers hold.  `rank`'s own rows [*o0, *o1) and window [*w0, *w1): x = 0 level-0 image rows into the image buffers;
// x = j or L-1+j (backward), j = 1 .. L-1, cumulative flow of level L-j into the cum_in rows of level L-1-j; x = 2L-1
// level-0 backward total rows into the rows the check holds.
static void exchange_rows(const StripPlan &pl, int x, int rank, int *o0, int *o1, int *w0, int *w1)
{
    const int L = pl.levels;
    if (x == 0 || x == 2 * L - 1) {
        const LevelStrip s = pl.strips(rank)[0];
        *o0 = s.y0, *o1 = s.y1;
        if (x == 0) *w0 = s.eb0, *w1 = s.eb1;
        else pl.fb_rows(rank, w0, w1);
        return;
    }
    const int j = x < L ? x : x - (L - 1);
    const LevelStrip own = pl.level(L - j, rank), fine = pl.level(L - 1 - j, rank);
    *o0 = own.y0, *o1 = own.y1, *w0 = fine.cy0, *w1 = fine.cy1;
}
// Rows [lo, hi) of one exchange between this rank and `peer`; the receiving rank's buffer starts at global row `base`.
struct HaloRows {
    int peer, lo, hi, base;
};
// The halo-row table of one rank, per exchange x in [0, nx) (numbering: ArenaLayout): the rows it sends and receives,
// the ranks it pushes to in either kind of pair (they acknowledge through done[], the teardown drains them) and the
// ranks that push to it (told at the end of a pair that their rows have been used; the check-row senders first, so
// that the handshake kernel's flags keep their order).
struct HaloTable {
    std::vector<std::vector<HaloRows>> send, recv;
    std::vector<int> done_from, sources;
};
static void add_unique(std::vector<int> &v, int x)
{
    if (std::find(v.begin(), v.end(), x) == v.end()) v.push_back(x);
}
// Sender and receiver lists come from the same exchange_rows, so they agree; the backward exchanges repeat the forward
// ones.  Every window holds its rank's own rows and both ends of a window grow with the rank, so the peers of an
// exchange are a run of ranks around `rank`: the scan stops at the first rank either side that shares no rows.
static HaloTable halo_table(const StripPlan &pl, int nx, int rank)
{
    HaloTable t;
    t.send.assign(nx, {});
    t.recv.assign(nx, {});
    for (int x = 0; x < nx; x++) {
        int m0, m1, mw0, mw1;
        exchange_rows(pl, x, rank, &m0, &m1, &mw0, &mw1);
        auto shares = [&](int peer, bool add) {
            int p0, p1, pw0, pw1;
            exchange_rows(pl, x, peer, &p0, &p1, &pw0, &pw1);
            // my own rows in the peer's window, and the peer's own rows in mine
            const int s0 = std::max(m0, pw0), s1 = std::min(m1, pw1), r0 = std::max(p0, mw0), r1 = std::min(p1, mw1);
            if (add && s0 < s1) t.send[x].push_back({peer, s0, s1, pw0});
            if (add && r0 < r1) t.recv[x].push_back({peer, r0, r1, mw0});
            return s0 < s1 || r0 < r1;
        };
        int first = rank, last = rank;
        while (first > 0 && shares(first - 1, false)) first--;
        while (last + 1 < pl.world && shares(last + 1, false)) last++;
        for (int peer = first; peer <= last; peer++)
            if (peer != rank) shares(peer, true);
        for (const HaloRows &e : t.send[x]) add_unique(t.done_from, e.peer);
    }
    if (nx > pl.levels)
        for (const HaloRows &e : t.recv[nx - 1]) add_unique(t.sources, e.peer);
    for (int x = 0; x < nx; x++)
        for (const HaloRows &e : t.recv[x]) add_unique(t.sources, e.peer);
    return t;
}

struct PeerSeg {
    const void *src;
    void *dst; // inside a peer's arena
    size_t bytes; // multiple of 8
};
struct PeerPushArgs {
    PeerSeg seg[PEER_MAX_SEG];
    int nseg, ndst;
    unsigned *arrive[PEER_MAX_DST];           // arrive[x * world + me] in the arena of each destination
    const unsigned *done_local[PEER_MAX_DST]; // done[dst] in MY arena: dst has finished with what I pushed last pair
    unsigned *counter;                        // counter[x] in my arena
    const unsigned *pairs;                    // pairs completed (my arena): this pair's epoch is *pairs + 1
    int *err;
};
struct PeerWaitArgs {
    const unsigned *flag[PEER_MAX_DST]; // arrive[x * world + src] in my arena
    int n;
    const unsigned *pairs;
    int *err;
};
struct PeerDoneArgs {
    unsigned *flag[2 * PEER_MAX_DST]; // done[me] in the arena of every rank that pushes to me
    int n;
    unsigned *pairs;
};
constexpr unsigned long long PEER_TIMEOUT_NS = 4000000000ull; // a peer that never shows up: flag the pair, do not hang

__device__ __forceinline__ unsigned long long peer_now()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ unsigned peer_ld(const unsigned *p)
{
    unsigned v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
// true when *p has reached `epoch` (wrap-safe), false after PEER_TIMEOUT_NS
__device__ bool peer_spin(const unsigned *p, unsigned epoch)
{
    const unsigned long long t0 = peer_now();
    while ((int)(peer_ld(p) - epoch) < 0) {
        if (peer_now() - t0 > PEER_TIMEOUT_NS) return false;
        __nanosleep(100);
    }
    return true;
}

// Sender side of one exchange: wait until every destination has finished with last pair's rows, store the segments into
// the destinations' arenas (peer stores over NVLink), and -- last block out -- raise the epoch flag in each of them.
__global__ void __launch_bounds__(256) peer_push_kernel(const __grid_constant__ PeerPushArgs a)
{
    const unsigned epoch = *a.pairs + 1u;
    if (threadIdx.x < a.ndst && !peer_spin(a.done_local[threadIdx.x], epoch - 1u)) atomicOr(a.err, 2);
    __syncthreads();
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x, nt = (size_t)gridDim.x * blockDim.x;
    for (int s = 0; s < a.nseg; s++) {
        const PeerSeg g = a.seg[s];
        if (((reinterpret_cast<uintptr_t>(g.src) | reinterpret_cast<uintptr_t>(g.dst) | g.bytes) & 15) == 0) {
            const uint4 *src = static_cast<const uint4 *>(g.src);
            uint4 *dst = static_cast<uint4 *>(g.dst);
            for (size_t i = t; i < g.bytes / 16; i += nt) dst[i] = src[i];
        } else {
            const uint2 *src = static_cast<const uint2 *>(g.src);
            uint2 *dst = static_cast<uint2 *>(g.dst);
            for (size_t i = t; i < g.bytes / 8; i += nt) dst[i] = src[i];
        }
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned arrived = atomicAdd(a.counter, 1u);
        if (arrived == gridDim.x - 1) {
            *a.counter = 0u;
            __threadfence_system();
            for (int d = 0; d < a.ndst; d++) asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(a.arrive[d]), "r"(epoch) : "memory");
        }
    }
}
// Receiver side: one thread per source spins on its epoch flag.
__global__ void peer_wait_kernel(const __grid_constant__ PeerWaitArgs a)
{
    if (threadIdx.x < a.n && !peer_spin(a.flag[threadIdx.x], *a.pairs + 1u)) atomicOr(a.err, 2);
    __threadfence_system();
}
// Teardown: wait until every rank this one pushed to has acknowledged this rank's last pair (done[dst] == pairs).
struct PeerDrainArgs {
    const unsigned *flag[2 * PEER_MAX_DST];
    int n;
    const unsigned *pairs;
    int *err;
};
__global__ void peer_drain_kernel(const __grid_constant__ PeerDrainArgs a)
{
    if (threadIdx.x < a.n && !peer_spin(a.flag[threadIdx.x], *a.pairs)) atomicOr(a.err, 2);
}
// End of a pair: tell every rank that pushes to me that its rows have been used, and count the pair.
__global__ void peer_done_kernel(const __grid_constant__ PeerDoneArgs a)
{
    const unsigned epoch = *a.pairs + 1u;
    if (threadIdx.x < a.n) asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(a.flag[threadIdx.x]), "r"(epoch) : "memory");
    __syncthreads();
    if (threadIdx.x == 0) *a.pairs = epoch;
}
} // namespace ofb

using namespace ofb;

#define OFB_STRIPS_GUARD(st)                       \
    DeviceGuard _guard(ctx_device((st)->ctx));     \
    if (!_guard.ok) return OFB_ERR_CUDA

struct ofb_strips {
    ofb_ctx *ctx = nullptr;
    StripPlan plan;
    int rank = 0, warp_mode = OFB_WARP_BILINEAR;
    float flow_scale = 1.0f;
    std::vector<LevelStrip> s;                 // this rank's strip per level
    // the halo-row table, per exchange x in [0, lay.nx) (numbering: ArenaLayout): rows this rank sends and receives
    std::vector<std::vector<HaloRows>> send, recv;
    std::vector<size_t> pitch;                 // image pitch per level
    std::vector<uint8_t *> prev, next;         // [eb0, eb1) rows
    std::vector<float *> flow, cum, cum_in;    // flow / cum: buffer rows (origin eb0); cum_in[k]: rows [cy0, cy1) of cum_{k+1}
    std::vector<size_t> img_stride;            // next[k] - prev[k]: both frames of a level are one batch of two images
    std::vector<float *> cum_dst;              // where level k's kernel writes its cumulative flow (buffer-row indexing like
                                               // flow[k]): straight into cum_in[k-1], whose rows [cy0, cy1) contain the own rows
    int want_total = 1;                        // level 0 also writes its cumulative flow (the total flow of the pair)
    int fused = 1;                             // cumulative-flow halo rows are pushed by the level kernels themselves
    int *overflow = nullptr;
    std::vector<void *> allocs;
    // peer memory
    uint8_t *arena = nullptr;               // my arena (one cudaMalloc: prev[0], next[0], cum_in[], flags live in it)
    ArenaLayout lay;
    std::vector<uint8_t *> peer_arena;      // base of every rank's arena in this process's address space (nullptr: not mapped)
    std::vector<ArenaLayout> peer_lay;
    std::vector<void *> ipc_opened;
    bool peers_connected = false;
    std::vector<int> done_from;             // ranks this one pushes to: they write done[rank] into this arena (teardown waits for it)
    std::vector<int> sources;               // ranks that push to this one, in a pair of either kind: told when their rows are used
    // checked pairs (ofb_strips_create_fb): the backward direction's buffers, laid out like the forward ones
    std::vector<float *> flow_b, cum_in_b, cum_dst_b; // cum_dst_b[0]: level 0's rows inside fbh
    float *fbh = nullptr;                   // backward total flow, rows [hy0, hy1) of level 0 (in the arena)
    int hy0 = 0, hy1 = 0;
    uint8_t *status = nullptr;              // own rows [y0, y1) of level 0
    float *err2 = nullptr;
};

namespace {
int dev_alloc(ofb_strips *st, void **p, size_t bytes)
{
    OFB_CUDA_TRY(cudaMalloc(p, bytes ? bytes : 16));
    OFB_CUDA_TRY(cudaMemset(*p, 0, bytes ? bytes : 16));
    st->allocs.push_back(*p);
    return OFB_OK;
}
// pixels of the own rows of level 0
inline size_t s_own_px(const ofb_strips *st) { return (size_t)st->s[0].w * (st->s[0].y1 - st->s[0].y0); }

// ---- peer memory: one exchange ---------------------------------------------------------------------------------------
struct PeerSend {
    int peer;
    const void *src;
    size_t dst_off; // in the peer's arena
    size_t bytes;
};
inline unsigned *flag_ptr(uint8_t *arena, const ArenaLayout &lay, size_t index)
{
    return reinterpret_cast<unsigned *>(arena + lay.flags) + index;
}
// Exchange x of the pair: push `sends`, then wait for the ranks this one receives rows from (recv[x]).
// (do_push / do_wait: the two halves, which ofb_strips_run_phase_device enqueues separately.)
int peer_exchange(ofb_strips *st, int x, const std::vector<PeerSend> &sends, cudaStream_t q, unsigned long long *launches, bool do_push,
                  bool do_wait)
{
    const int me = st->rank;
    unsigned *pairs = flag_ptr(st->arena, st->lay, st->lay.pairs());
    if (do_push && !sends.empty()) {
        PeerPushArgs a{};
        size_t total = 0;
        for (const PeerSend &sd : sends) {
            if (a.nseg == PEER_MAX_SEG || !st->peer_arena[sd.peer]) {
                set_error("strips: exchange %d has too many segments or an unmapped peer %d (strips thinner than the halo?)", x, sd.peer);
                return OFB_ERR_UNSUPPORTED;
            }
            a.seg[a.nseg++] = PeerSeg{sd.src, st->peer_arena[sd.peer] + sd.dst_off, sd.bytes};
            total += sd.bytes;
            bool seen = false;
            for (int d = 0; d < a.ndst; d++) seen |= a.arrive[d] == flag_ptr(st->peer_arena[sd.peer], st->peer_lay[sd.peer], st->peer_lay[sd.peer].arrive(x, me));
            if (!seen) {
                if (a.ndst == PEER_MAX_DST) {
                    set_error("strips: exchange %d sends to more than %d ranks", x, PEER_MAX_DST);
                    return OFB_ERR_UNSUPPORTED;
                }
                a.arrive[a.ndst] = flag_ptr(st->peer_arena[sd.peer], st->peer_lay[sd.peer], st->peer_lay[sd.peer].arrive(x, me));
                a.done_local[a.ndst] = flag_ptr(st->arena, st->lay, st->lay.done(sd.peer));
                a.ndst++;
            }
        }
        a.counter = flag_ptr(st->arena, st->lay, st->lay.counter(x));
        a.pairs = pairs;
        a.err = st->overflow;
        const unsigned blocks = (unsigned)std::min<size_t>(64, std::max<size_t>(1, total / (256 * 64)));
        peer_push_kernel<<<blocks, 256, 0, q>>>(a);
        OFB_CUDA_TRY(cudaGetLastError());
        if (launches) ++*launches;
    }
    if (do_wait && !st->recv[x].empty()) {
        PeerWaitArgs w{};
        for (const HaloRows &e : st->recv[x]) {
            if (w.n == PEER_MAX_DST) {
                set_error("strips: exchange %d receives from more than %d ranks", x, PEER_MAX_DST);
                return OFB_ERR_UNSUPPORTED;
            }
            w.flag[w.n++] = flag_ptr(st->arena, st->lay, st->lay.arrive(x, e.peer));
        }
        w.pairs = pairs;
        w.err = st->overflow;
        peer_wait_kernel<<<1, 32, 0, q>>>(w);
        OFB_CUDA_TRY(cudaGetLastError());
        if (launches) ++*launches;
    }
    return OFB_OK;
}
// The schedule of a w x h pair of `levels` levels cut into `world` strips (arguments checked by the caller); refuses a
// coarsest level with fewer rows than strips, and strips so thin that some rank's halo rows come from, or go to, more
// ranks than one exchange carries (PEER_MAX_DST ranks, PEER_MAX_SEG copy segments; 2 PEER_MAX_DST ranks in the
// end-of-pair handshake).  The table of EVERY rank is checked, so that every rank refuses the same plan: a rank whose own
// exchanges fit must not go on alone into the peer set-up.
int make_plan(int w, int h, int levels, int win, int world, int reach, int fb_reach, StripPlan *pl)
{
    const int hc = h >> (levels - 1);
    if (hc < world || (w >> (levels - 1)) < 1) {
        set_error("coarsest level has %d rows, cannot cut it into %d strips", hc, world);
        return OFB_ERR_INVALID;
    }
    pl->W = w, pl->H = h, pl->levels = levels, pl->win = win, pl->world = world, pl->reach = reach;
    pl->fb_reach = fb_reach;
    pl->r = win / 2;
    // image halo: 3x3 stencil + window radius + one row of even-row alignment + warp reach + bilinear tap
    pl->img_halo = pl->r + 2 + reach + 2;
    const int nx = fb_reach >= 0 ? 2 * levels : levels;
    for (int rank = 0; rank < world; rank++) {
        HaloTable t;
        try { // (std::vector growth must not throw across the C ABI)
            t = halo_table(*pl, nx, rank);
        } catch (const std::bad_alloc &) {
            set_error("strips: out of host memory");
            return OFB_ERR_NOMEM;
        }
        // (what is over the limit, the exchange or -1 for the whole pair, the count, the limit)
        const char *what = nullptr;
        int x = -1, n = 0, limit = 0;
        for (int e = 0; e < nx && !what; e++) {
            if ((n = (int)t.send[e].size()) > PEER_MAX_DST) what = "sends rows to %d ranks", x = e, limit = PEER_MAX_DST;
            else if ((n = (int)t.recv[e].size()) > PEER_MAX_DST) what = "receives rows from %d ranks", x = e, limit = PEER_MAX_DST;
        }
        if (!what && (n = 2 * (int)t.send[0].size()) > PEER_MAX_SEG) what = "copies %d segments", x = 0, limit = PEER_MAX_SEG;
        if (!what && (n = (int)t.sources.size()) > 2 * PEER_MAX_DST) what = "receives rows from %d ranks", limit = 2 * PEER_MAX_DST;
        if (!what && (n = (int)t.done_from.size()) > 2 * PEER_MAX_DST) what = "sends rows to %d ranks", limit = 2 * PEER_MAX_DST;
        if (what) {
            char ex[40] = "the exchanges of a pair", msg[64];
            if (x >= 0) snprintf(ex, sizeof ex, "exchange %d", x);
            snprintf(msg, sizeof msg, what, n);
            set_error("strips thinner than their halo: in %s rank %d %s, more than the limit of %d; use fewer ranks, fewer levels "
                      "or a smaller reach / fb_reach", ex, rank, msg, limit);
            return OFB_ERR_UNSUPPORTED;
        }
    }
    return OFB_OK;
}
} // namespace

extern "C" {

// The strip schedule as this library computes it, without a device: rows of `level` on `rank` as
// out8 = {y0, y1, by0, by1, cy0, cy1, eb0, eb1} (own rows; rows the level kernel needs; rows of the next-coarser
// cumulative flow held; rows the image buffers hold, which adds what building the coarser levels' halo rows locally
// takes).  Lets a host check its own partitioning -- and the tests check cuda_optical_flow_2_b200/dist.py -- against it.
int ofb_strips_plan_query(int w, int h, int levels, int win, int world, int rank, int reach, int level, int *out8)
{
    if (!out8 || w < 1 || h < 1 || levels < 1 || levels > OFB_MAX_LEVELS || (win & 1) == 0 || win < 3 || win > OFB_MAX_WINDOW ||
        world < 1 || rank < 0 || rank >= world || reach < 0 || level < 0 || level >= levels) {
        set_error("strips_plan_query: bad arguments");
        return OFB_ERR_INVALID;
    }
    StripPlan pl;
    if (int rc = make_plan(w, h, levels, win, world, reach, -1, &pl)) return rc;
    const LevelStrip s = pl.strips(rank)[level];
    const int v[8] = {s.y0, s.y1, s.by0, s.by1, s.cy0, s.cy1, s.eb0, s.eb1};
    memcpy(out8, v, sizeof v);
    return OFB_OK;
}

} // extern "C"

// ofb_strips_create (fb_reach < 0) and ofb_strips_create_fb
static int strips_create_impl(ofb_ctx *ctx, int w, int h, int levels, int win, int warp_mode, float flow_scale, int world, int rank,
                              int reach, int fb_reach, ofb_strips **out)
{
    if (!ctx || !out || w < 1 || h < 1 || levels < 1 || levels > OFB_MAX_LEVELS || (win & 1) == 0 || win < 3 ||
        win > OFB_MAX_WINDOW || world < 1 || rank < 0 || rank >= world || reach < 0) {
        set_error("strips_create: bad arguments");
        return OFB_ERR_INVALID;
    }
    if (warp_mode == OFB_WARP_AS_WRITTEN && levels > 1) {
        set_error("OFB_WARP_AS_WRITTEN needs pixel (0,0) of every coarser level: not available on strips");
        return OFB_ERR_UNSUPPORTED;
    }
    StripPlan pl;
    if (int rc = make_plan(w, h, levels, win, world, reach, fb_reach, &pl)) return rc;
    DeviceGuard guard(ctx_device(ctx));
    if (!guard.ok) return OFB_ERR_CUDA;
    ofb_strips *st = new (std::nothrow) ofb_strips;
    if (!st) {
        set_error("strips_create: out of host memory");
        return OFB_ERR_NOMEM;
    }
    try { // (std::vector growth below must not throw across the C ABI)
    st->ctx = ctx;
    st->rank = rank;
    st->warp_mode = warp_mode;
    st->flow_scale = flow_scale;
    st->plan = pl;
    int rc = OFB_OK;
    st->s = pl.strips(rank);
    // what neighbours write into (level-0 image rows, coarser cumulative-flow rows, flags): one allocation, the arena
    st->lay = arena_layout(pl, rank);
    {
        HaloTable t = halo_table(pl, st->lay.nx, rank);
        st->send = std::move(t.send);
        st->recv = std::move(t.recv);
        st->done_from = std::move(t.done_from);
        st->sources = std::move(t.sources);
    }
    {
        void *p = nullptr;
        rc = dev_alloc(st, &p, st->lay.bytes);
        st->arena = static_cast<uint8_t *>(p);
    }
    for (int k = 0; k < levels && rc == OFB_OK; k++) {
        const LevelStrip s = st->s[k];
        const size_t pitch = ((size_t)s.w + 63) / 64 * 64;
        st->pitch.push_back(pitch);
        void *p = nullptr;
        const int rows = s.eb1 - s.eb0;
        if (k == 0) {
            st->prev.push_back(st->arena + st->lay.prev0);
            st->next.push_back(st->arena + st->lay.next0);
            st->img_stride.push_back(st->lay.next0 - st->lay.prev0);
        } else { // one block: the pyramid step handles prev and next as a batch of two
            const size_t stride = (pitch * rows + 255) / 256 * 256;
            if ((rc = dev_alloc(st, &p, 2 * stride))) break;
            st->prev.push_back(static_cast<uint8_t *>(p));
            st->next.push_back(static_cast<uint8_t *>(p) + stride);
            st->img_stride.push_back(stride);
        }
        if ((rc = dev_alloc(st, &p, (size_t)s.w * rows * 8))) break;
        st->flow.push_back(static_cast<float *>(p));
        // the cumulative flow of level 0 (the total flow) has its own buffer; levels >= 1 write theirs straight into the
        // buffer the next finer level reads (below), whose other rows the neighbours fill
        p = nullptr;
        if (k == 0 && (rc = dev_alloc(st, &p, (size_t)s.w * rows * 8))) break;
        st->cum.push_back(static_cast<float *>(p));
        st->cum_in.push_back(reinterpret_cast<float *>(st->arena + st->lay.cum_in[k]));
    }
    if (fb_reach >= 0) {
        pl.fb_rows(rank, &st->hy0, &st->hy1);
        st->fbh = reinterpret_cast<float *>(st->arena + st->lay.fbh);
        const size_t own = s_own_px(st);
        void *p = nullptr;
        if (rc == OFB_OK) rc = dev_alloc(st, &p, own);
        st->status = static_cast<uint8_t *>(p);
        p = nullptr;
        if (rc == OFB_OK) rc = dev_alloc(st, &p, own * 4);
        st->err2 = static_cast<float *>(p);
        for (int k = 0; k < levels && rc == OFB_OK; k++) {
            const LevelStrip s = st->s[k];
            if ((rc = dev_alloc(st, &p, (size_t)s.w * (s.eb1 - s.eb0) * 8))) break;
            st->flow_b.push_back(static_cast<float *>(p));
            st->cum_in_b.push_back(reinterpret_cast<float *>(st->arena + st->lay.cum_in_b[k]));
        }
        for (int k = 0; k < levels && rc == OFB_OK; k++) {
            const LevelStrip &s = st->s[k];
            st->cum_dst_b.push_back(k == 0 ? st->fbh + ((ptrdiff_t)s.eb0 - st->hy0) * (ptrdiff_t)s.w * 2
                                           : st->cum_in_b[k - 1] + ((ptrdiff_t)s.eb0 - st->s[k - 1].cy0) * (ptrdiff_t)s.w * 2);
        }
    }
    for (int k = 0; k < levels && rc == OFB_OK; k++) {
        // buffer row b of level k is global row eb0 + b; row g of cum_in[k-1] sits at (g - cy0) * w
        float *dst = st->cum[k];
        if (k > 0) {
            const LevelStrip &s = st->s[k], &fine = st->s[k - 1];
            dst = st->cum_in[k - 1] + ((ptrdiff_t)s.eb0 - fine.cy0) * (ptrdiff_t)s.w * 2;
            if (s.y0 < fine.cy0 || s.y1 > fine.cy1) {
                set_error("strips_create: level %d own rows [%d,%d) outside the finer level's coarse window [%d,%d)", k, s.y0, s.y1,
                          fine.cy0, fine.cy1);
                rc = OFB_ERR_INVALID;
            }
        }
        st->cum_dst.push_back(dst);
    }
    if (rc == OFB_OK) {
        void *p = nullptr;
        rc = dev_alloc(st, &p, sizeof(int));
        st->overflow = static_cast<int *>(p);
    }
    // every kernel a pair launches is loaded now: a lazily loaded kernel may synchronise the context at its first
    // launch, which must not happen behind a kernel that waits for a neighbour
    if (rc == OFB_OK) rc = preload_lk_level(win);
    if (rc == OFB_OK) rc = preload_pyramid();
    if (rc == OFB_OK && fb_reach >= 0) rc = preload_fb_check_strip();
    if (rc == OFB_OK) {
        cudaFuncAttributes fa;
        if (cudaFuncGetAttributes(&fa, peer_push_kernel) != cudaSuccess || cudaFuncGetAttributes(&fa, peer_wait_kernel) != cudaSuccess ||
            cudaFuncGetAttributes(&fa, peer_done_kernel) != cudaSuccess) {
            set_error("strips_create: loading the exchange kernels failed");
            rc = OFB_ERR_CUDA;
        }
    }
    if (rc == OFB_OK && cudaDeviceSynchronize() != cudaSuccess) { // the zeroed flags must be in place before a peer can see the arena
        set_error("strips_create: device synchronisation failed");
        rc = OFB_ERR_CUDA;
    }
    if (rc != OFB_OK) {
        for (void *p : st->allocs) cudaFree(p);
        delete st;
        return rc;
    }
    } catch (const std::bad_alloc &) {
        for (void *p : st->allocs) cudaFree(p);
        delete st;
        set_error("strips_create: out of host memory");
        return OFB_ERR_NOMEM;
    }
    *out = st;
    return OFB_OK;
}

extern "C" {

int ofb_strips_create(ofb_ctx *ctx, int w, int h, int levels, int win, int warp_mode, float flow_scale, int world, int rank,
                      int reach, ofb_strips **out)
{
    return strips_create_impl(ctx, w, h, levels, win, warp_mode, flow_scale, world, rank, reach, -1, out);
}

int ofb_strips_create_fb(ofb_ctx *ctx, int w, int h, int levels, int win, int warp_mode, float flow_scale, int world, int rank,
                         int reach, int fb_reach, ofb_strips **out)
{
    if (fb_reach < 0 || !(std::isfinite(flow_scale) && flow_scale > 0.0f)) {
        set_error("strips_create_fb: fb_reach %d must be >= 0 and flow_scale %g finite and > 0", fb_reach, (double)flow_scale);
        return OFB_ERR_INVALID;
    }
    return strips_create_impl(ctx, w, h, levels, win, warp_mode, flow_scale, world, rank, reach, fb_reach, out);
}

// ---- peer memory: set-up ----------------------------------------------------------------------------------------
// The 128-byte blob a rank publishes: its arena's CUDA IPC handle and the arena's offset inside the allocation the
// handle stands for (small cudaMalloc blocks share one).
int ofb_strips_peer_handle(ofb_strips *st, void *blob128)
{
    if (!st || !blob128) {
        set_error("strips_peer_handle: bad arguments");
        return OFB_ERR_INVALID;
    }
    OFB_STRIPS_GUARD(st);
    memset(blob128, 0, 128);
    cudaIpcMemHandle_t h;
    OFB_CUDA_TRY(cudaIpcGetMemHandle(&h, st->arena));
    static_assert(sizeof h == 64, "CUDA IPC handle size");
    memcpy(blob128, &h, sizeof h);
    unsigned long long off = 0;
    {
        typedef int (*GetRange)(unsigned long long *, size_t *, unsigned long long);
        void *sym = nullptr;
        cudaDriverEntryPointQueryResult q;
        unsigned long long base = 0;
        size_t size = 0;
        if (cudaGetDriverEntryPoint("cuMemGetAddressRange", &sym, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess && sym &&
            reinterpret_cast<GetRange>(sym)(&base, &size, (unsigned long long)reinterpret_cast<uintptr_t>(st->arena)) == 0)
            off = (unsigned long long)reinterpret_cast<uintptr_t>(st->arena) - base;
        else {
            set_error("strips_peer_handle: cuMemGetAddressRange failed");
            return OFB_ERR_CUDA;
        }
    }
    memcpy(static_cast<char *>(blob128) + 64, &off, sizeof off);
    return OFB_OK;
}

int ofb_strips_peer_arena(ofb_strips *st, void **arena)
{
    if (!st || !arena) {
        set_error("strips_peer_arena: bad arguments");
        return OFB_ERR_INVALID;
    }
    *arena = st->arena;
    return OFB_OK;
}

namespace {
// ranks whose buffers I write into, or that write into mine, at any exchange
bool is_neighbour(const ofb_strips *st, int peer)
{
    return std::find(st->done_from.begin(), st->done_from.end(), peer) != st->done_from.end() ||
           std::find(st->sources.begin(), st->sources.end(), peer) != st->sources.end();
}
int finish_connect(ofb_strips *st)
{
    st->peer_lay.clear();
    for (int peer = 0; peer < st->plan.world; peer++) st->peer_lay.push_back(arena_layout(st->plan, peer));
    st->peers_connected = true;
    return OFB_OK;
}
} // namespace

// blobs: world x 128 bytes, rank r's ofb_strips_peer_handle blob at 128 * r (an all-gather by the application).
int ofb_strips_peer_connect(ofb_strips *st, const void *blobs)
{
    if (!st || !blobs) {
        set_error("strips_peer_connect: bad arguments");
        return OFB_ERR_INVALID;
    }
    OFB_STRIPS_GUARD(st);
    const int world = st->plan.world;
    st->peer_arena.assign(world, nullptr);
    st->peer_arena[st->rank] = st->arena;
    for (int peer = 0; peer < world; peer++) {
        if (peer == st->rank || !is_neighbour(st, peer)) continue;
        cudaIpcMemHandle_t h;
        unsigned long long off = 0;
        memcpy(&h, static_cast<const char *>(blobs) + 128 * (size_t)peer, sizeof h);
        memcpy(&off, static_cast<const char *>(blobs) + 128 * (size_t)peer + 64, sizeof off);
        void *base = nullptr;
        OFB_CUDA_TRY(cudaIpcOpenMemHandle(&base, h, cudaIpcMemLazyEnablePeerAccess));
        st->ipc_opened.push_back(base);
        st->peer_arena[peer] = static_cast<uint8_t *>(base) + off;
    }
    return finish_connect(st);
}

// Same, for ranks that live in ONE process (tests; a single-process multi-GPU host with peer access enabled by the
// caller): arenas[r] = ofb_strips_peer_arena of rank r.
int ofb_strips_peer_connect_local(ofb_strips *st, void *const *arenas)
{
    if (!st || !arenas) {
        set_error("strips_peer_connect_local: bad arguments");
        return OFB_ERR_INVALID;
    }
    st->peer_arena.assign(st->plan.world, nullptr);
    for (int peer = 0; peer < st->plan.world; peer++) st->peer_arena[peer] = static_cast<uint8_t *>(arenas[peer]);
    st->peer_arena[st->rank] = st->arena;
    return finish_connect(st);
}

// Teardown.  The last thing a neighbour writes into this rank's arena is its `done` flag at the end of its last pair,
// which can land after this rank has finished its own: so, before the arena is unmapped and freed, wait (on the device,
// bounded like every other wait) until every rank this one pushes to has acknowledged this rank's last pair.  Ranks must
// have run the same number of pairs; a rank that is still PUSHING a further pair into a freed arena is a caller error.
int ofb_strips_destroy(ofb_strips *st)
{
    if (!st) return OFB_OK;
    {
        DeviceGuard guard(ctx_device(st->ctx));
        if (guard.ok) {
            cudaDeviceSynchronize();
            if (st->plan.world > 1 && st->peers_connected && !st->done_from.empty()) {
                PeerDrainArgs d{};
                for (int dst : st->done_from)
                    if (d.n < 2 * PEER_MAX_DST) d.flag[d.n++] = flag_ptr(st->arena, st->lay, st->lay.done(dst));
                d.pairs = flag_ptr(st->arena, st->lay, st->lay.pairs());
                d.err = st->overflow;
                peer_drain_kernel<<<1, 32>>>(d);
                cudaDeviceSynchronize();
            }
            for (void *p : st->ipc_opened) cudaIpcCloseMemHandle(p);
            for (void *p : st->allocs) cudaFree(p);
        }
    }
    delete st;
    return OFB_OK;
}

int ofb_strips_own_rows(const ofb_strips *st, int level, int *y0, int *y1)
{
    if (!st || level < 0 || level >= st->plan.levels) {
        set_error("strips_own_rows: bad arguments");
        return OFB_ERR_INVALID;
    }
    if (y0) *y0 = st->s[level].y0;
    if (y1) *y1 = st->s[level].y1;
    return OFB_OK;
}

int ofb_strips_result(const ofb_strips *st, int level, float **flow_own_d, float **total_own_d)
{
    if (!st || level < 0 || level >= st->plan.levels) {
        set_error("strips_result: bad arguments");
        return OFB_ERR_INVALID;
    }
    const LevelStrip &s = st->s[level];
    const size_t off = (size_t)(s.y0 - s.eb0) * s.w * 2;
    if (flow_own_d) *flow_own_d = st->flow[level] + off;
    // cumulative flow exists where a level writes it: every level but the coarsest (whose cumulative flow is its flow)
    if (total_own_d) *total_own_d = (st->plan.levels == 1 ? st->flow[level] : st->cum_dst[level]) + off;
    return OFB_OK;
}

// Where the own rows [y0, y1) of level 0 live: a producer that writes them there and passes the same pointers to
// ofb_strips_run_device saves the upload copy.
int ofb_strips_input(const ofb_strips *st, uint8_t **prev_own_d, uint8_t **next_own_d, size_t *pitch)
{
    if (!st) {
        set_error("strips_input: NULL handle");
        return OFB_ERR_INVALID;
    }
    const LevelStrip &s = st->s[0];
    const size_t off = (size_t)(s.y0 - s.eb0) * st->pitch[0];
    if (prev_own_d) *prev_own_d = st->prev[0] + off;
    if (next_own_d) *next_own_d = st->next[0] + off;
    if (pitch) *pitch = st->pitch[0];
    return OFB_OK;
}

// Whether level 0 also writes the total (cumulative) flow of the pair; on by default, 8 more bytes per pixel.
int ofb_strips_set_total(ofb_strips *st, int on)
{
    if (!st) {
        set_error("strips_set_total: NULL handle");
        return OFB_ERR_INVALID;
    }
    st->want_total = on ? 1 : 0;
    return OFB_OK;
}

// Whether the cumulative-flow halo rows are pushed by the level kernels themselves (default) or by separate copy / wait
// kernels (for comparison).
int ofb_strips_set_fused(ofb_strips *st, int on)
{
    if (!st) {
        set_error("strips_set_fused: NULL handle");
        return OFB_ERR_INVALID;
    }
    st->fused = on ? 1 : 0;
    return OFB_OK;
}

} // extern "C"

namespace {
// The coarse-to-fine level loop of one direction of a pair: forward (prev -> next) or, in a checked pair, backward
// (next -> prev on the same pyramid, with its own residual-flow buffers, cum_in regions and exchanges).  Level k's
// neighbours' cumulative-flow rows arrive by exchange xb + L - 1 - k; the loop's phases start at pb (see
// strips_run_impl).  In the backward loop of a checked pair level 0 writes the backward total into fbh, and -- fused
// form, at most two targets -- its kernel also pushes the rows the neighbours' checks need (*check_pushed).
int strips_levels(ofb_strips *st, bool bwd, bool checked, cudaStream_t q, int phase, bool *check_pushed,
                  unsigned long long *launches)
{
    auto on = [phase](int ph) { return phase < 0 || phase == ph; };
    const StripPlan &pl = st->plan;
    const bool peer_mode = pl.world > 1;
    const int L = pl.levels, me = st->rank;
    const int pb = bwd ? 2 * L - 1 : 0, xb = bwd ? L - 1 : 0;
    const std::vector<float *> &flow = bwd ? st->flow_b : st->flow, &cum_in = bwd ? st->cum_in_b : st->cum_in;
    const std::vector<float *> &cum_dst = bwd ? st->cum_dst_b : st->cum_dst;
    auto peer_cum_in = [&](int peer, int k) { return bwd ? st->peer_lay[peer].cum_in_b[k] : st->peer_lay[peer].cum_in[k]; };
    // coarse to fine: rows [cy0, cy1) of cum_{k+1} into cum_in[k] (own part copied, the rest received), then the level
    bool pushed_by_kernel = false; // the exchange that feeds the level at hand was pushed by the previous (coarser) level's kernel
    for (int k = L - 1; k >= 0; k--) {
        const LevelStrip &s = st->s[k];
        const int j = L - 1 - k, x = xb + j; // this level's step of the loop, and the exchange that feeds it
        bool wait_in_kernel = false;
        if (k < L - 1) {
            const LevelStrip &up = st->s[k + 1];
            // level k+1 wrote its own rows of cum_{k+1} straight into cum_in[k] (cum_dst); the neighbours' rows follow
            const float *src = cum_dst[k + 1]; // buffer-row indexing of level k+1 (origin up.eb0)
            const size_t rowf = (size_t)up.w * 2;  // floats per row
            if (peer_mode) {
                std::vector<PeerSend> sends;
                for (const HaloRows &e : st->send[x])
                    sends.push_back({e.peer, src + (size_t)(e.lo - up.eb0) * rowf, peer_cum_in(e.peer, k) + (size_t)(e.lo - e.base) * rowf * 4,
                                     (size_t)(e.hi - e.lo) * rowf * 4});
                // Fused form: level k+1's kernel has already pushed my rows (pushed_by_kernel, previous iteration) and this
                // level's kernel waits for the neighbours' flags itself; the copy / wait kernels remain for what does not
                // fit the kernel's two slots (strips thinner than the halo).
                wait_in_kernel = st->fused && !st->recv[x].empty() && st->recv[x].size() <= 2;
                int rc = peer_exchange(st, x, sends, q, launches, on(pb + 2 * j) && !pushed_by_kernel, on(pb + 2 * j + 1) && !wait_in_kernel);
                if (rc) return rc;
            }
        }
        // what THIS level's kernel pushes: my rows of cum_k that the neighbours' level k-1 needs (exchange x + 1), or, at
        // level 0 of the backward loop of a checked pair, my rows of the backward total their checks need (2L - 1)
        LkLevelArgs::PeerPush push[2] = {};
        int npush = 0;
        const int xn = k >= 1 ? x + 1 : 2 * L - 1;
        pushed_by_kernel = false;
        if (peer_mode && st->fused && (k >= 1 || (bwd && checked)) && !st->send[xn].empty() && st->send[xn].size() <= 2) {
            for (const HaloRows &e : st->send[xn]) {
                const ArenaLayout &pa = st->peer_lay[e.peer];
                push[npush].dst = reinterpret_cast<float *>(st->peer_arena[e.peer] + (k >= 1 ? peer_cum_in(e.peer, k - 1) : pa.fbh)) +
                                  ((ptrdiff_t)s.eb0 - e.base) * (ptrdiff_t)s.w * 2;
                push[npush].row_lo = e.lo - s.eb0;
                push[npush].row_hi = e.hi - s.eb0;
                push[npush].flag = flag_ptr(st->peer_arena[e.peer], pa, pa.arrive(xn, me));
                push[npush].done = flag_ptr(st->arena, st->lay, st->lay.done(e.peer));
                npush++;
            }
            pushed_by_kernel = true;
        }
        if (k == 0 && bwd) *check_pushed = pushed_by_kernel;
        if (!on(pb + 2 * j + 1)) continue;
        LkLevelArgs a = lk_args_strip(bwd ? st->next[k] : st->prev[k], bwd ? st->prev[k] : st->next[k], st->pitch[k], s.w, s.eb1 - s.eb0,
                                      s.eb0, s.h, s.y0 - s.eb0, s.y1 - s.eb0, pl.win, st->warp_mode, st->flow_scale, flow[k],
                                      ctx_sm_count(st->ctx), ctx_solve_fast(st->ctx));
        a.cum_in = k < L - 1 ? cum_in[k] : nullptr;
        a.cum_w = s.w >> 1;
        a.cum_h_global = s.h >> 1;
        a.cum_y_off = s.cy0;
        a.cum_h_local = std::max(s.cy1 - s.cy0, 1);
        // every level but the finest feeds the next one; level 0 writes the total flow (always in a checked pair)
        const bool want_cum = k > 0 || checked || (L > 1 && st->want_total);
        a.cum_out = want_cum ? cum_dst[k] : nullptr;
        a.reach_overflow = st->overflow;
        if (npush > 0 && a.cum_out) {
            a.npush = npush;
            a.push[0] = push[0];
            a.push[1] = push[1];
            a.push_counter = flag_ptr(st->arena, st->lay, st->lay.fused(xn));
        }
        if (wait_in_kernel) {
            const std::vector<HaloRows> &rv = st->recv[x];
            a.nwait = (int)rv.size();
            for (int d = 0; d < a.nwait; d++)
                a.wait[d] = {flag_ptr(st->arena, st->lay, st->lay.arrive(x, rv[d].peer)), rv[d].lo - s.cy0, rv[d].hi - s.cy0};
        }
        a.epoch_src = flag_ptr(st->arena, st->lay, st->lay.pairs());
        int rc = launch_lk_level(a, q, launches);
        if (rc) return rc;
    }
    return OFB_OK;
}
} // namespace

// One pair: own rows of level 0 in, residual (and cumulative) flow of the own rows of every level out, all
// asynchronous on `stream`.  prev_own_d / next_own_d: rows [y0, y1) of level 0, planar u8 with `pitch` bytes per row.
// fb != NULL: a checked pair (handles of ofb_strips_create_fb): the backward level loop on the same pyramid, the exchange
// of the backward total rows the neighbours' checks sample, and the check of the own rows.
//
// `phase` < 0: the whole pair.  Otherwise one of its phases, so that a host can interleave the ranks of ONE process on ONE
// stream in an order in which no kernel ever waits for a later one:
//   phase 0      own-row upload, push of the level-0 image rows (exchange 0)
//   phase 1      wait for exchange 0, pyramid, coarsest level L-1
//   phase 2j     push of the cumulative-flow rows of level L-j (exchange j),            j = 1 .. L-1
//   phase 2j+1   wait for exchange j, level L-1-j; after level 0 of a plain pair the end-of-pair handshake
// and in a checked pair (4L + 1 phases):
//   phase 2L         backward coarsest level L-1
//   phase 2L+2j-1    push of the backward cumulative-flow rows of level L-j (exchange L-1+j), j = 1 .. L-1
//   phase 2L+2j      wait for exchange L-1+j, backward level L-1-j
//   phase 4L-1       push of the backward total rows the neighbours' checks sample (exchange 2L-1)
//   phase 4L         wait for exchange 2L-1, the check, the end-of-pair handshake
struct FbRun {
    float alpha, beta;
    int want_err2;
};
static int strips_run_impl(ofb_strips *st, const uint8_t *prev_own_d, const uint8_t *next_own_d, size_t pitch, void *stream, int phase,
                           const FbRun *fb = nullptr)
{
    if (!st || !prev_own_d || !next_own_d) {
        set_error("strips_run: bad arguments");
        return OFB_ERR_INVALID;
    }
    if (fb && st->plan.fb_reach < 0) {
        set_error("strips_run_fb: the handle was not created by ofb_strips_create_fb");
        return OFB_ERR_INVALID;
    }
    if (fb && !(std::isfinite(fb->alpha) && fb->alpha >= 0.0f && std::isfinite(fb->beta) && fb->beta >= 0.0f)) {
        set_error("strips_run_fb: alpha %g / beta %g must be finite and >= 0", (double)fb->alpha, (double)fb->beta);
        return OFB_ERR_INVALID;
    }
    OFB_STRIPS_GUARD(st);
    try { // (std::vector growth must not throw across the C ABI)
    auto on = [phase](int ph) { return phase < 0 || phase == ph; };
    cudaStream_t q = static_cast<cudaStream_t>(stream);
    const StripPlan &pl = st->plan;
    const bool peer_mode = pl.world > 1;
    if (peer_mode && !st->peers_connected) {
        set_error("strips_run: world > 1 and the peers are not connected (call ofb_strips_peer_connect first)");
        return OFB_ERR_INVALID;
    }
    const int L = pl.levels, me = st->rank;
    const int nphase = fb ? 4 * L + 1 : 2 * L;
    if (phase >= nphase) {
        set_error("strips_run_phase: phase %d of %d", phase, nphase);
        return OFB_ERR_INVALID;
    }
    unsigned long long *launches = ctx_launch_counter(st->ctx);
    if (pitch < (size_t)pl.W) {
        set_error("strips_run: pitch %zu smaller than the width %d", pitch, pl.W);
        return OFB_ERR_INVALID;
    }
    if (on(0)) {
        const LevelStrip &s = st->s[0];
        const size_t off = (size_t)(s.y0 - s.eb0) * st->pitch[0];
        // a producer that wrote the own rows in place (ofb_strips_input) saves this copy
        if (prev_own_d != st->prev[0] + off)
            OFB_CUDA_TRY(cudaMemcpy2DAsync(st->prev[0] + off, st->pitch[0], prev_own_d, pitch, (size_t)s.w, (size_t)(s.y1 - s.y0),
                                           cudaMemcpyDeviceToDevice, q));
        if (next_own_d != st->next[0] + off)
            OFB_CUDA_TRY(cudaMemcpy2DAsync(st->next[0] + off, st->pitch[0], next_own_d, pitch, (size_t)s.w, (size_t)(s.y1 - s.y0),
                                           cudaMemcpyDeviceToDevice, q));
    }
    // (the error flag st->overflow is sticky: kernels OR into it, only ofb_strips_check clears it)
    // ONE image exchange, on level 0: the rows of my buffer that other ranks own (and vice versa), in place
    const int eb0 = st->s[0].eb0;
    const size_t P = st->pitch[0];
    if (peer_mode) {
        std::vector<PeerSend> sends;
        for (const HaloRows &e : st->send[0]) {
            const ArenaLayout &pa = st->peer_lay[e.peer];
            sends.push_back({e.peer, st->prev[0] + (size_t)(e.lo - eb0) * P, pa.prev0 + (size_t)(e.lo - e.base) * P, (size_t)(e.hi - e.lo) * P});
            sends.push_back({e.peer, st->next[0] + (size_t)(e.lo - eb0) * P, pa.next0 + (size_t)(e.lo - e.base) * P, (size_t)(e.hi - e.lo) * P});
        }
        int rc = peer_exchange(st, 0, sends, q, launches, on(0), on(1));
        if (rc) return rc;
    }
    // pyramid: every buffer row of level k+1 from the buffer rows of level k (halo rows are built locally)
    for (int k = 0; on(1) && k + 1 < L; k++) {
        const LevelStrip &s = st->s[k], &d = st->s[k + 1];
        int rc = launch_pyr_down_strip(st->prev[k], st->pitch[k], s.w, s.eb1 - s.eb0, s.eb0, st->prev[k + 1], st->pitch[k + 1], d.eb0,
                                       d.eb1, q, launches, 2, st->img_stride[k], st->img_stride[k + 1]);
        if (rc) return rc;
    }
    bool check_pushed = false;
    int rc = strips_levels(st, false, fb != nullptr, q, phase, &check_pushed, launches);
    if (rc) return rc;
    if (fb) {
        if ((rc = strips_levels(st, true, true, q, phase, &check_pushed, launches))) return rc;
        // exchange 2L-1: my own rows of the backward total that the neighbours' checks sample (unless level 0's kernel pushed
        // them), then the wait for the rows I sample
        if (peer_mode) {
            const LevelStrip &s = st->s[0];
            const size_t rowf = (size_t)s.w * 2;
            std::vector<PeerSend> sends;
            for (const HaloRows &e : st->send[2 * L - 1])
                sends.push_back({e.peer, st->fbh + (size_t)(e.lo - st->hy0) * rowf, st->peer_lay[e.peer].fbh + (size_t)(e.lo - e.base) * rowf * 4,
                                 (size_t)(e.hi - e.lo) * rowf * 4});
            if ((rc = peer_exchange(st, 2 * L - 1, sends, q, launches, on(4 * L - 1) && !check_pushed, on(4 * L))))
                return rc;
        }
        if (on(4 * L)) {
            const LevelStrip &s = st->s[0];
            if ((rc = launch_fb_check_strip(st->cum[0] + (size_t)(s.y0 - s.eb0) * s.w * 2, st->fbh, s.w, s.h, s.y0, s.y1 - s.y0, st->hy0,
                                            st->hy1, st->flow_scale, fb->alpha, fb->beta, st->status, fb->want_err2 ? st->err2 : nullptr,
                                            st->overflow, q, launches)))
                return rc;
        }
    }
    if (peer_mode && on(nphase - 1)) { // the rows my neighbours pushed have been used: they may push the next pair's
        PeerDoneArgs d{};
        for (int src : st->sources) {
            if (d.n == 2 * PEER_MAX_DST) {
                set_error("strips: more than %d ranks push to this one", 2 * PEER_MAX_DST);
                return OFB_ERR_UNSUPPORTED;
            }
            d.flag[d.n++] = flag_ptr(st->peer_arena[src], st->peer_lay[src], st->peer_lay[src].done(me));
        }
        d.pairs = flag_ptr(st->arena, st->lay, st->lay.pairs());
        peer_done_kernel<<<1, 32, 0, q>>>(d);
        OFB_CUDA_TRY(cudaGetLastError());
        if (launches) ++*launches;
    }
    } catch (const std::bad_alloc &) {
        set_error("strips_run: out of host memory");
        return OFB_ERR_NOMEM;
    }
    return OFB_OK;
}

extern "C" {

int ofb_strips_run_device(ofb_strips *st, const uint8_t *prev_own_d, const uint8_t *next_own_d, size_t pitch, void *stream)
{
    return strips_run_impl(st, prev_own_d, next_own_d, pitch, stream, -1);
}

int ofb_strips_run_phase_device(ofb_strips *st, const uint8_t *prev_own_d, const uint8_t *next_own_d, size_t pitch, int phase,
                                void *stream)
{
    if (phase < 0) {
        set_error("strips_run_phase: phase %d", phase);
        return OFB_ERR_INVALID;
    }
    return strips_run_impl(st, prev_own_d, next_own_d, pitch, stream, phase);
}

int ofb_strips_run_fb_device(ofb_strips *st, const uint8_t *prev_own_d, const uint8_t *next_own_d, size_t pitch, float alpha, float beta,
                             int want_err2, void *stream)
{
    const FbRun fb{alpha, beta, want_err2};
    return strips_run_impl(st, prev_own_d, next_own_d, pitch, stream, -1, &fb);
}

int ofb_strips_run_fb_phase_device(ofb_strips *st, const uint8_t *prev_own_d, const uint8_t *next_own_d, size_t pitch, float alpha,
                                   float beta, int want_err2, int phase, void *stream)
{
    if (phase < 0) {
        set_error("strips_run_fb_phase: phase %d", phase);
        return OFB_ERR_INVALID;
    }
    const FbRun fb{alpha, beta, want_err2};
    return strips_run_impl(st, prev_own_d, next_own_d, pitch, stream, phase, &fb);
}

int ofb_strips_fb_result(const ofb_strips *st, float **fwd_total_own_d, float **bwd_total_own_d, uint8_t **status_own_d,
                         float **err2_own_d)
{
    if (!st || st->plan.fb_reach < 0) {
        set_error("strips_fb_result: NULL handle, or one not created by ofb_strips_create_fb");
        return OFB_ERR_INVALID;
    }
    const LevelStrip &s = st->s[0];
    if (fwd_total_own_d) *fwd_total_own_d = st->cum[0] + (size_t)(s.y0 - s.eb0) * s.w * 2;
    if (bwd_total_own_d) *bwd_total_own_d = st->fbh + (size_t)(s.y0 - st->hy0) * s.w * 2;
    if (status_own_d) *status_own_d = st->status;
    if (err2_own_d) *err2_own_d = st->err2;
    return OFB_OK;
}

// Synchronises the stream and reports whether a warp sample reached past the exchanged halo rows (the result is
// then NOT the whole-frame result: raise `reach`).
int ofb_strips_check(ofb_strips *st, void *stream, int *overflow)
{
    if (!st) {
        set_error("strips_check: NULL handle");
        return OFB_ERR_INVALID;
    }
    OFB_STRIPS_GUARD(st);
    int v = 0;
    // sticky flag: everything since the last check; read, then clear (in stream order, so pairs enqueued later start clean)
    OFB_CUDA_TRY(cudaMemcpyAsync(&v, st->overflow, sizeof(int), cudaMemcpyDeviceToHost, static_cast<cudaStream_t>(stream)));
    OFB_CUDA_TRY(cudaMemsetAsync(st->overflow, 0, sizeof(int), static_cast<cudaStream_t>(stream)));
    OFB_CUDA_TRY(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
    if (overflow) *overflow = v;
    return OFB_OK;
}

} // extern "C"
