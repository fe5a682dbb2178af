// lk_win.cu -- the fused per-level LK kernels of ONE window size (-DLK_WIN=n): grid sizing and the
// (warp mode, cumulative output) dispatch.  See lk_level.cu for the entry point.
#include "lk_level.cuh"

#include <algorithm>
#include <climits>
#include <cstdlib>

#ifndef LK_WIN
#error "compile with -DLK_WIN=<odd window 3..19>"
#endif

namespace ofb {

int lk_make_image_map(CUtensorMap *tm, const uint8_t *base, int w, int h, int n, size_t pitch, size_t stride, int box_w,
                      int box_rows);
int lk_make_flow_map(CUtensorMap *tm, const float *base, int w, int h, int n, size_t pair_stride_vec, int box_w, int box_rows,
                     int *usable);

template <int WIN, int MODE, bool CUMOUT, bool FAST, bool PEER, bool COMP>
static int launch_one(const LkLevelArgs &a, cudaStream_t stream, unsigned long long *launches)
{
    using C = LkCfg<WIN>;
    static bool attr_set[64] = {};
    int dev = 0;
    OFB_CUDA_TRY(cudaGetDevice(&dev));
    if (dev < 64 && !attr_set[dev]) {
        OFB_CUDA_TRY(cudaFuncSetAttribute(lk_level_kernel<WIN, MODE, CUMOUT, FAST, PEER, COMP>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          C::smem_bytes(FAST, CUMOUT && MODE != 0)));
        attr_set[dev] = true;
    }
    CUtensorMap tmP, tmQ;
    int rc = lk_make_image_map(&tmP, a.prev, a.w, a.h_local, a.n_pairs, a.pitch, a.image_stride, LK_TILE_W, C::CH);
    if (rc) return rc;
    // next: the same box as prev on the coarsest level, the window with margin on warped levels
    rc = lk_make_image_map(&tmQ, a.next, a.w, a.h_local, a.n_pairs, a.pitch, a.image_stride, MODE != 0 ? LK_NTW : LK_TILE_W,
                           MODE != 0 ? C::NTH : C::CH);
    if (rc) return rc;
    // coarser cumulative flow of bilinearly warped levels: tiles of NBR x LK_CTW vectors
    CUtensorMap tmC = tmP;
    int cum_tma = 0;
    if (MODE != 0) {
        rc = lk_make_flow_map(&tmC, a.cum_in, a.cum_w, a.cum_h_local, a.n_pairs, a.cum_pair_stride, LK_CTW, C::NBR, &cum_tma);
        if (rc) return rc;
    }

    CUtensorMap tmC2 = tmP;
    if (COMP) {
        int usable = 0;
        rc = lk_make_flow_map(&tmC2, a.cum2_in, a.cum_w >> 1, a.cum_h_global >> 1, a.n_pairs, a.cum2_pair_stride, LK_C2W, C::NBR / 2 + 1,
                              &usable);
        if (rc) return rc;
        if (!usable || !cum_tma) {
            set_error("lk_level: composition on the fly needs 16-byte aligned coarser flow rows (caller checks lk_can_compose)");
            return OFB_ERR_INVALID;
        }
    }

    const int out_rows = a.out_y1 - a.out_y0;
    const int strips = (a.w + C::TWO - 1) / C::TWO;
    // Rows per CTA.  The hardware hands CTAs to SMs as slots free up, so a launch takes about
    // (total row-steps) / SMs plus a ragged tail of roughly half a CTA's lifetime (MIN_BLOCKS CTAs
    // share an SM, so a CTA lives MIN_BLOCKS times its own row-steps).  Short CTAs shrink the tail,
    // tall CTAs amortise the 2R+2 halo rows: take the split that minimises the sum.
    const int n_sm = a.sm_count > 0 ? a.sm_count : 148;
    const long long cols = (long long)strips * a.n_pairs;
    const int max_ny = (out_rows + C::CH - 1) / C::CH;
    int rows_per_block = out_rows;
    double best = 1e300;
    for (int ny = 1; ny <= max_ny && ny <= 128; ny++) {
        const int rpb = (out_rows + ny - 1) / ny;
        const int nb = (out_rows + rpb - 1) / rpb;
        // rows a CTA processes: its outputs plus the 2R+2 halo rows (+1 for the even first row), rounded up to
        // whole sub-chunks by the V/H phases and to whole chunks by the gather (about a quarter of the work)
        const int need = rpb + 2 * C::R + 3;
        const double steps = 0.75 * ((need + C::SUB - 1) / C::SUB * C::SUB) + 0.25 * ((need + C::CH - 1) / C::CH * C::CH);
        const double cost = (double)(cols * nb) * steps / n_sm + 0.5 * C::MIN_BLOCKS * steps;
        if (cost < best * 0.999) {
            best = cost;
            rows_per_block = rpb;
        }
    }
    if (const char *dbg = getenv("OFB_LK_ROWS")) { // developer override for experiments
        const int v = atoi(dbg);
        if (v > 0) rows_per_block = v < out_rows ? v : out_rows;
    }
    const int nby = (out_rows + rows_per_block - 1) / rows_per_block;
    // A big batch of full-height CTAs drains for a whole CTA lifetime while the SMs run emptier and emptier (one 1080p
    // column strip lives ~0.3 ms, 3 % of a 1024-pair launch).  The last wave's worth of pairs is therefore cut into 4 row
    // blocks each: a quarter of the drain for 11 halo rows more per block on those pairs only.
    int tail_pair0 = INT_MAX, tail_shift = 0, tail_rows = 0, grid_z = a.n_pairs;
    {
        const char *env = getenv("OFB_LK_TAIL"); // developer override: 0 = off, n = 2^n row blocks per tail pair
        const char *envw = getenv("OFB_LK_TAIL_WAVES"); // ... and the length of the tail in tenths of a wave
        const int shift = env ? atoi(env) : 2;
        const int slots = n_sm * C::MIN_BLOCKS;
        int tail_pairs = ((slots + strips - 1) / strips * (envw ? atoi(envw) : 10) + 9) / 10;
        // grid z = n + ((1 << shift) - 1) * tail_pairs must stay within the hardware's 65535: near that many pairs the
        // tail shrinks, and at 65535 it is off
        if (shift > 0 && shift <= 4) tail_pairs = std::min(tail_pairs, (65535 - a.n_pairs) / ((1 << shift) - 1));
        if (shift > 0 && shift <= 4 && nby == 1 && a.npush == 0 && a.nwait == 0 && out_rows >= (2 * C::CH << shift) &&
            tail_pairs > 0 && (long long)a.n_pairs * strips >= 4ll * slots && tail_pairs < a.n_pairs) {
            tail_shift = shift;
            tail_pair0 = a.n_pairs - tail_pairs;
            tail_rows = (out_rows + (1 << shift) - 1) >> shift;
            grid_z = tail_pair0 + (tail_pairs << tail_shift);
        }
    }

    LkKernelParams p;
    p.next = a.next;
    p.pitch = (int)a.pitch;
    p.image_stride = a.image_stride;
    p.w = a.w;
    p.h_local = a.h_local;
    p.y_off = a.y_off;
    p.h_global = a.h_global;
    p.out_y0 = a.out_y0;
    p.out_y1 = a.out_y1;
    p.rows_per_block = rows_per_block;
    p.tail_pair0 = tail_pair0;
    p.tail_shift = tail_shift;
    p.tail_rows = tail_rows;
    p.as_written = (a.warp_mode == OFB_WARP_AS_WRITTEN) ? 1 : 0;
    p.scale2 = 2.0f * a.flow_scale;
    p.scale512 = 512.0f * a.flow_scale;
    p.cum_in = reinterpret_cast<const float2 *>(a.cum_in);
    p.cum_w = a.cum_w;
    p.cum_h_global = a.cum_h_global;
    p.cum_y_off = a.cum_y_off;
    p.cum_h_local = a.cum_h_local;
    p.cum_pair_stride = a.cum_pair_stride;
    p.flow_out = reinterpret_cast<float2 *>(a.flow_out);
    p.cum_out = reinterpret_cast<float2 *>(a.cum_out);
    p.flow_pair_stride = a.flow_pair_stride;
    p.reach_overflow = a.reach_overflow;
    p.cum_tma = cum_tma;
    p.cum2_in = reinterpret_cast<const float2 *>(a.cum2_in);
    p.cum2_w = a.cum_w >> 1;
    p.cum2_pair_stride = a.cum2_pair_stride;
    p.npush = a.npush;
    p.nwait = a.nwait;
    p.push_counter = a.push_counter;
    p.epoch_src = a.epoch_src;
    for (int d = 0; d < 2; d++) {
        p.push[d] = LkPeerPush{};
        p.wait[d] = LkPeerWait{};
        if (d < a.npush) {
            // CTAs of this launch that own rows of [row_lo, row_hi): every column strip of every row block that meets it
            unsigned blocks = 0;
            for (int b = 0; b < nby; b++) {
                const int ys = a.out_y0 + b * rows_per_block, ye = std::min(ys + rows_per_block, a.out_y1);
                if (ys < a.push[d].row_hi && ye > a.push[d].row_lo) blocks++;
            }
            p.push[d] = LkPeerPush{reinterpret_cast<float2 *>(a.push[d].dst), a.push[d].row_lo, a.push[d].row_hi, a.push[d].flag,
                                   a.push[d].done, blocks * (unsigned)strips};
            if (blocks == 0 || a.n_pairs != 1) {
                set_error("lk_level: fused halo push needs one pair and rows inside the launch (rows [%d,%d))", a.push[d].row_lo,
                          a.push[d].row_hi);
                return OFB_ERR_INVALID;
            }
        }
        if (d < a.nwait) p.wait[d] = LkPeerWait{a.wait[d].flag, a.wait[d].crow_lo, a.wait[d].crow_hi};
    }

    dim3 grid((unsigned)strips, (unsigned)nby, (unsigned)grid_z);
    OFB_CUDA_TRY(launch_pdl(lk_level_kernel<WIN, MODE, CUMOUT, FAST, PEER, COMP>, grid, dim3(LK_NT), C::smem_bytes(FAST, CUMOUT && MODE != 0),
                            stream, tmP, tmQ, tmC, tmC2, p));
    if (launches) ++*launches;
    return OFB_OK;
}

template <int WIN, bool FAST, bool PEER> static int launch_lk_win_solve(const LkLevelArgs &a, cudaStream_t s, unsigned long long *l)
{
    const bool co = a.cum_out != nullptr;
    if (a.cum_in == nullptr)
        return co ? launch_one<WIN, 0, true, FAST, PEER, false>(a, s, l) : launch_one<WIN, 0, false, FAST, false, false>(a, s, l);
    if (!PEER && a.cum2_in != nullptr) { // the coarser level's cumulative flow composed on the fly
        if (a.warp_mode == OFB_WARP_BILINEAR)
            return co ? launch_one<WIN, 2, true, FAST, false, true>(a, s, l) : launch_one<WIN, 2, false, FAST, false, true>(a, s, l);
        return co ? launch_one<WIN, 1, true, FAST, false, true>(a, s, l) : launch_one<WIN, 1, false, FAST, false, true>(a, s, l);
    }
    if (a.warp_mode == OFB_WARP_BILINEAR)
        return co ? launch_one<WIN, 2, true, FAST, PEER, false>(a, s, l) : launch_one<WIN, 2, false, FAST, PEER, false>(a, s, l);
    return co ? launch_one<WIN, 1, true, FAST, PEER, false>(a, s, l) : launch_one<WIN, 1, false, FAST, PEER, false>(a, s, l);
}
template <int WIN> int launch_lk_win(const LkLevelArgs &a, cudaStream_t s, unsigned long long *l)
{
    const bool peer = a.npush > 0 || a.nwait > 0;
    if (peer) return a.solve_fast ? launch_lk_win_solve<WIN, true, true>(a, s, l) : launch_lk_win_solve<WIN, false, true>(a, s, l);
    return a.solve_fast ? launch_lk_win_solve<WIN, true, false>(a, s, l) : launch_lk_win_solve<WIN, false, false>(a, s, l);
}

template int launch_lk_win<LK_WIN>(const LkLevelArgs &a, cudaStream_t s, unsigned long long *l);

// Loads every variant of this window's kernel now (CUDA loads kernels lazily, and loading may synchronise the context:
// a launch that first has to load its kernel can then not be enqueued behind a kernel that spins on a neighbour).
template <int WIN, bool FAST, bool PEER> static int preload_lk_win_solve()
{
    cudaFuncAttributes fa;
    if (!PEER) OFB_CUDA_TRY(cudaFuncGetAttributes(&fa, lk_level_kernel<WIN, 0, false, FAST, false, false>));
    OFB_CUDA_TRY(cudaFuncGetAttributes(&fa, lk_level_kernel<WIN, 0, true, FAST, PEER, false>));
    OFB_CUDA_TRY(cudaFuncGetAttributes(&fa, lk_level_kernel<WIN, 1, false, FAST, PEER, false>));
    OFB_CUDA_TRY(cudaFuncGetAttributes(&fa, lk_level_kernel<WIN, 1, true, FAST, PEER, false>));
    OFB_CUDA_TRY(cudaFuncGetAttributes(&fa, lk_level_kernel<WIN, 2, false, FAST, PEER, false>));
    OFB_CUDA_TRY(cudaFuncGetAttributes(&fa, lk_level_kernel<WIN, 2, true, FAST, PEER, false>));
    if (!PEER) {
        OFB_CUDA_TRY(cudaFuncGetAttributes(&fa, lk_level_kernel<WIN, 1, false, FAST, false, true>));
        OFB_CUDA_TRY(cudaFuncGetAttributes(&fa, lk_level_kernel<WIN, 1, true, FAST, false, true>));
        OFB_CUDA_TRY(cudaFuncGetAttributes(&fa, lk_level_kernel<WIN, 2, false, FAST, false, true>));
        OFB_CUDA_TRY(cudaFuncGetAttributes(&fa, lk_level_kernel<WIN, 2, true, FAST, false, true>));
    }
    return OFB_OK;
}
template <int WIN> int preload_lk_win()
{
    int rc = preload_lk_win_solve<WIN, false, false>();
    if (!rc) rc = preload_lk_win_solve<WIN, true, false>();
    if (!rc) rc = preload_lk_win_solve<WIN, false, true>();
    if (!rc) rc = preload_lk_win_solve<WIN, true, true>();
    return rc;
}
template int preload_lk_win<LK_WIN>();

} // namespace ofb
