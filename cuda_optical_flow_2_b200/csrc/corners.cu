// corners.cu -- Shi-Tomasi corner detection for the point tracker (ofb_min_eig_map_device, ofb_detect_corners_device; the
// rule is pinned in include/ofb200.h).  The score of a pixel is the tracker's own texture measure: the smaller eigenvalue
// of the exact int32 structure tensor of the tracker's level-0 Sobel fields over the window, over win^2, computed in
// double with every operation rounded on its own, so that the kernel and the tests' C restatement (tests/corner_oracle.c)
// agree bit for bit.
//
// Five steps per call, all on the caller's stream and none of them waiting on the host:
//   corner_init_kernel     per image: interior maximum 0, candidate segment [i*cap, i*cap)
//   corner_score_kernel    the hot path: a 32 x 32 tile per CTA, its bytes plus a win/2 + 1 halo staged in shared memory,
//                          Sobel fields as int16, sliding column sums and then sliding row sums of the three products in
//                          int32, the score in double; the interior maximum through an integer atomicMax on the float bits
//                          (scores are >= 0, so the maximum does not depend on the order)
//   corner_cand_kernel     the threshold and the 3x3 key-order test; a candidate's key (~score_bits << 32 | raster index)
//                          is appended to its image's segment (the order inside a segment is fixed by the sort)
//   cub sort               ascending keys per image = strongest first, ties in raster order (corner_sort_bytes)
//   corner_select_kernel   one CTA per image: the sequential greedy of the rule, a chunk of keys at a time (below)
#include "ofb_common.cuh"

#include <cub/block/block_scan.cuh>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_segmented_sort.cuh>

namespace ofb {

constexpr int CRN_TW = 32, CRN_TH = 32, CRN_THREADS = 256; // score tile and CTA
constexpr int CRN_SEG = 8;                                   // rows per thread in the column-sum pass
constexpr int SEL_CHUNK = 512;                               // keys per step of the selection (= its CTA size)
constexpr int SEL_WORDS = SEL_CHUNK / 32;

template <int WIN> struct CrnCfg {
    static constexpr int R = WIN / 2;
    static constexpr int FW = CRN_TW + 2 * R, FH = CRN_TH + 2 * R; // field positions the tile's windows cover
    static constexpr int BW = FW + 2, BH = FH + 2;                 // staged bytes
    static constexpr int CS = (FW + 3) / 4 * 4 + 1;                // column-sum row stride: == 1 (mod 4), no bank conflicts
};

// The score of one window from its exact sums (include/ofb200.h): the stable form of (S - sqrt(disc)) / 2 in double, every
// operation rounded on its own (no fma), then / win^2 and rounded to float.
__device__ __forceinline__ float crn_score(int A, int D, int B, double win2)
{
    const int S = A + D;
    if (S == 0) return 0.0f;
    const long long det = (long long)A * D - (long long)B * B, T = (long long)A - D;
    const long long disc = T * T + 4 * (long long)B * B;
    const double l1 = __ddiv_rn(__dmul_rn(2.0, __ll2double_rn(det)), __dadd_rn((double)S, __dsqrt_rn(__ll2double_rn(disc))));
    return __double2float_rn(__ddiv_rn(l1, win2));
}

template <int WIN>
__global__ void __launch_bounds__(CRN_THREADS) corner_score_kernel(const CornerArgs a)
{
    using C = CrnCfg<WIN>;
    constexpr int R = C::R, FW = C::FW, FH = C::FH, BW = C::BW, BH = C::BH, CS = C::CS;
    __shared__ uint8_t s_b[BH * BW];
    __shared__ int16_t s_gx[FH * FW], s_gy[FH * FW];
    __shared__ int s_ca[CRN_TH * CS], s_cd[CRN_TH * CS], s_cb[CRN_TH * CS];
    const int t = threadIdx.x, z = blockIdx.z;
    const uint8_t *img = a.img + (size_t)z * a.istr;
    // (grid.y is capped at 65535; ty * CRN_TH would overflow int past the last tile of a frame taller than 2^31 - 2^21)
    for (int ty = blockIdx.y; ty <= (a.h - 1) / CRN_TH; ty += gridDim.y) {
        const int x0 = blockIdx.x * CRN_TW, y0 = ty * CRN_TH; // the tile's first output pixel
        // bytes of (x0 - R - 1, y0 - R - 1) .. + (BW, BH); 0 outside the frame
        for (int i = t; i < BH * BW; i += CRN_THREADS) {
            const int r = i / BW, c = i - r * BW, x = x0 - R - 1 + c, y = y0 - R - 1 + r;
            s_b[i] = (x >= 0 && x < a.w && y >= 0 && y < a.h) ? __ldg(img + (size_t)y * a.pitch + x) : (uint8_t)0;
        }
        __syncthreads();
        // Sobel fields at (x0 - R + c, y0 - R + r); 0 at positions outside the frame
        for (int i = t; i < FH * FW; i += CRN_THREADS) {
            const int r = i / FW, c = i - r * FW, x = x0 - R + c, y = y0 - R + r;
            int gx = 0, gy = 0;
            if (x >= 0 && x < a.w && y >= 0 && y < a.h) {
                const uint8_t *q = s_b + r * BW + c;
                const int p00 = q[0], p01 = q[1], p02 = q[2], p10 = q[BW], p12 = q[BW + 2];
                const int p20 = q[2 * BW], p21 = q[2 * BW + 1], p22 = q[2 * BW + 2];
                gx = (p02 + 2 * p12 + p22) - (p00 + 2 * p10 + p20);
                gy = (p20 + 2 * p21 + p22) - (p00 + 2 * p01 + p02);
            }
            s_gx[i] = (int16_t)gx;
            s_gy[i] = (int16_t)gy;
        }
        __syncthreads();
        // column sums over WIN field rows for output rows [seg*CRN_SEG, +CRN_SEG), sliding down
        for (int i = t; i < FW * (CRN_TH / CRN_SEG); i += CRN_THREADS) {
            const int c = i % FW, r0 = (i / FW) * CRN_SEG;
            int sa = 0, sd = 0, sb = 0;
#pragma unroll
            for (int k = 0; k < WIN; k++) {
                const int gx = s_gx[(r0 + k) * FW + c], gy = s_gy[(r0 + k) * FW + c];
                sa += gx * gx;
                sd += gy * gy;
                sb += gx * gy;
            }
#pragma unroll
            for (int r = 0; r < CRN_SEG; r++) {
                s_ca[(r0 + r) * CS + c] = sa;
                s_cd[(r0 + r) * CS + c] = sd;
                s_cb[(r0 + r) * CS + c] = sb;
                if (r + 1 < CRN_SEG) {
                    const int ox = s_gx[(r0 + r) * FW + c], oy = s_gy[(r0 + r) * FW + c];
                    const int nx = s_gx[(r0 + r + WIN) * FW + c], ny = s_gy[(r0 + r + WIN) * FW + c];
                    sa += nx * nx - ox * ox;
                    sd += ny * ny - oy * oy;
                    sb += nx * ny - ox * oy;
                }
            }
        }
        __syncthreads();
        // row sums over WIN column sums: thread = one row, 4 consecutive outputs, sliding right; then the score
        const int r = t >> 3, c0 = (t & 7) * 4, y = y0 + r;
        const double win2 = (double)(WIN * WIN);
        const int *ra = s_ca + r * CS, *rd = s_cd + r * CS, *rb = s_cb + r * CS;
        int sa = 0, sd = 0, sb = 0;
#pragma unroll
        for (int k = 0; k < WIN; k++) {
            sa += ra[c0 + k];
            sd += rd[c0 + k];
            sb += rb[c0 + k];
        }
        unsigned mx = 0;
        float *out = a.map + (size_t)z * a.map_stride + (size_t)y * a.w;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int x = x0 + c0 + j;
            const float s = crn_score(sa, sd, sb, win2);
            if (y < a.h && x < a.w) {
                out[x] = s;
                if (x >= a.m && x <= a.w - 1 - a.m && y >= a.m && y <= a.h - 1 - a.m) mx = max(mx, __float_as_uint(s));
            }
            if (j < 3) {
                sa += ra[c0 + j + WIN] - ra[c0 + j];
                sd += rd[c0 + j + WIN] - rd[c0 + j];
                sb += rb[c0 + j + WIN] - rb[c0 + j];
            }
        }
        if (a.max_bits) {
            mx = __reduce_max_sync(0xffffffffu, mx);
            if ((t & 31) == 0 && mx) atomicMax(a.max_bits + z, mx);
        }
        __syncthreads(); // the shared arrays before the next tile
    }
}

int launch_corner_score(const CornerArgs &a, int win, cudaStream_t stream, unsigned long long *launches)
{
    const dim3 grid((unsigned)((a.w - 1) / CRN_TW + 1), (unsigned)min((a.h - 1) / CRN_TH + 1, 65535), (unsigned)a.n);
    switch (win) {
#define OFB_CRN_CASE(W)                                                                   \
    case W: corner_score_kernel<W><<<grid, CRN_THREADS, 0, stream>>>(a); break;
        OFB_CRN_CASE(3)
        OFB_CRN_CASE(5)
        OFB_CRN_CASE(7)
        OFB_CRN_CASE(9)
        OFB_CRN_CASE(11)
        OFB_CRN_CASE(13)
        OFB_CRN_CASE(15)
        OFB_CRN_CASE(17)
        OFB_CRN_CASE(19)
#undef OFB_CRN_CASE
    default:
        set_error("corners: window %d not supported (odd 3..%d)", win, OFB_MAX_WINDOW);
        return OFB_ERR_UNSUPPORTED;
    }
    OFB_CUDA_TRY(cudaGetLastError());
    if (launches) ++*launches;
    return OFB_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// detection
// ---------------------------------------------------------------------------------------------------------------------
__global__ void corner_init_kernel(unsigned *max_bits, int *seg_begin, int *seg_end, int n, int cap)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        max_bits[i] = 0;
        seg_begin[i] = seg_end[i] = i * cap;
    }
}

// One thread per interior pixel (grid over the interior).  p precedes q: score(p) > score(q), or equal scores and p's raster
// index is the smaller; a candidate qualifies (score > thr) and precedes each of its interior 8-neighbours.
__global__ void __launch_bounds__(256) corner_cand_kernel(const float *__restrict__ map, size_t map_stride, int w, int h, int m,
                                                         const unsigned *__restrict__ max_bits, float quality_level,
                                                         float min_score, int *seg_end, unsigned long long *keys)
{
    const int z = blockIdx.z;
    const int x = m + blockIdx.x * 32 + threadIdx.x;
    const int x1 = w - 1 - m, y1 = h - 1 - m; // last interior column / row
    const float thr = fmaxf(__fmul_rn(quality_level, __uint_as_float(max_bits[z])), min_score);
    for (int y = m + blockIdx.y * 8 + threadIdx.y; y - threadIdx.y <= y1; y += gridDim.y * 8) { // (grid.y is capped at 65535)
        bool cand = false;
        float s = 0.0f;
        if (x <= x1 && y <= y1) {
            const float *row = map + (size_t)z * map_stride + (size_t)y * w + x;
            s = __ldg(row);
            if (s > thr) {
                cand = true;
#pragma unroll
                for (int dy = -1; dy <= 1; dy++)
#pragma unroll
                    for (int dx = -1; dx <= 1; dx++) {
                        if ((dx | dy) == 0) continue;
                        const int nx = x + dx, ny = y + dy;
                        if (nx < m || nx > x1 || ny < m || ny > y1) continue;
                        const float q = __ldg(row + (ptrdiff_t)dy * w + dx);
                        const bool earlier = dy < 0 || (dy == 0 && dx < 0); // the neighbour's raster index is smaller
                        cand &= earlier ? s > q : s >= q;
                    }
            }
        }
        const unsigned ball = __ballot_sync(0xffffffffu, cand); // a warp is one row
        if (!ball) continue;
        const int lane = threadIdx.x;
        int base = 0;
        if (lane == __ffs(ball) - 1) base = atomicAdd(seg_end + z, __popc(ball));
        base = __shfl_sync(0xffffffffu, base, __ffs(ball) - 1);
        if (cand)
            keys[base + __popc(ball & ((1u << lane) - 1))] =
                ((unsigned long long)(~__float_as_uint(s)) << 32) | (unsigned)(y * w + x);
    }
}

// One CTA per image, SEL_CHUNK keys at a time, in key order:
//   1. every key that conflicts with a corner accepted in an earlier chunk is dropped: a cell grid of side c (2 (c-1)^2 <
//      min_distance^2, so a cell holds at most one accepted corner) is looked up around it;
//   2. the survivors are compacted in key order and their pairwise conflicts (earlier survivor i, later j) set bit i of row
//      j of a bit matrix in shared memory;
//   3. rounds: an undecided survivor with an accepted earlier conflict is rejected, one with no undecided or accepted earlier
//      conflict is accepted.  The first undecided survivor always decides, so this ends, and it is the sequential greedy;
//      a chain of conflicts takes one round per link;
//   4. the accepted ones take the next output slots and enter the grid.
// Without suppression (min_distance^2 <= 1: distinct integer points are never closer than 1) every key is accepted.
struct SelArgs {
    const unsigned long long *keys; // sorted, image z's at [seg_begin[z], seg_end[z])
    const int *seg_begin, *seg_end;
    int w, m, max_corners;
    double md2;   // min_distance^2
    int suppress; // md2 > 1
    int cell, gw, gh, reach; // grid cell side, grid size (cells), the largest |dx| that can conflict
    int *grid;               // gw * gh per image, -1 = empty, else the raster index of the accepted corner
    float *corners, *scores;
    int *counts;
};

__global__ void __launch_bounds__(SEL_CHUNK) corner_select_kernel(const SelArgs a)
{
    using Scan = cub::BlockScan<int, SEL_CHUNK>;
    __shared__ typename Scan::TempStorage s_scan;
    __shared__ int s_x[SEL_CHUNK], s_y[SEL_CHUNK];
    __shared__ unsigned long long s_key[SEL_CHUNK];
    __shared__ unsigned s_conf[SEL_CHUNK][SEL_WORDS + 1]; // +1: the rows of one warp fall on different banks
    __shared__ unsigned s_acc[SEL_WORDS], s_und[SEL_WORDS];
    __shared__ int s_total;
    const int t = threadIdx.x, z = blockIdx.x, lane = t & 31, wid = t >> 5;
    // the chunk loop steps an offset inside the segment: a segment is at most one image's cap (< 2^29 keys), but it may end
    // anywhere below 2^31, where base + SEL_CHUNK would wrap
    const int begin = a.seg_begin[z], len = a.seg_end[z] - begin;
    int *grid = a.grid + (size_t)z * a.gw * a.gh;
    float2 *corners = reinterpret_cast<float2 *>(a.corners) + (size_t)z * a.max_corners;
    float *scores = a.scores ? a.scores + (size_t)z * a.max_corners : nullptr;
    int count = 0;
    for (int off = 0; off < len && count < a.max_corners; off += SEL_CHUNK) {
        bool alive = t < len - off;
        unsigned long long key = 0;
        int x = 0, y = 0;
        if (alive) {
            key = a.keys[begin + off + t];
            const int idx = (int)(unsigned)key;
            y = idx / a.w;
            x = idx - y * a.w;
        }
        if (alive && a.suppress) { // 1. the grid
            const int gx = x - a.m, gy = y - a.m;
            const int cx0 = max(0, gx - a.reach) / a.cell, cx1 = min(a.gw - 1, (gx + a.reach) / a.cell);
            const int cy0 = max(0, gy - a.reach) / a.cell, cy1 = min(a.gh - 1, (gy + a.reach) / a.cell);
            for (int cy = cy0; cy <= cy1 && alive; cy++)
                for (int cx = cx0; cx <= cx1; cx++) {
                    const int e = grid[cy * a.gw + cx];
                    if (e < 0) continue;
                    const int ey = e / a.w, ex = e - ey * a.w;
                    const long long dx = x - ex, dy = y - ey;
                    if ((double)(dx * dx + dy * dy) < a.md2) {
                        alive = false;
                        break;
                    }
                }
        }
        int pos, total; // 2. compaction in key order
        Scan(s_scan).ExclusiveSum(alive ? 1 : 0, pos, total);
        if (alive) {
            s_x[pos] = x;
            s_y[pos] = y;
            s_key[pos] = key;
        }
        __syncthreads();
        const bool mine = t < total;
        bool acc = mine;
        if (a.suppress && total > 1) {
            if (mine) {
                x = s_x[t];
                y = s_y[t];
                for (int wd = 0; wd <= t >> 5; wd++) {
                    unsigned bits = 0;
                    const int lim = min(32, t - 32 * wd);
                    for (int b = 0; b < lim; b++) {
                        const long long dx = x - s_x[32 * wd + b], dy = y - s_y[32 * wd + b];
                        if ((double)(dx * dx + dy * dy) < a.md2) bits |= 1u << b;
                    }
                    s_conf[t][wd] = bits;
                }
            }
            // 3. rounds; states: 0 undecided, 1 accepted, 2 rejected
            int st = mine ? 0 : 2;
            for (;;) {
                const unsigned und = __ballot_sync(0xffffffffu, st == 0), accb = __ballot_sync(0xffffffffu, st == 1);
                if (lane == 0) {
                    s_und[wid] = und;
                    s_acc[wid] = accb;
                }
                if (!__syncthreads_or(st == 0)) break;
                if (st == 0) {
                    bool hit_acc = false, hit_und = false;
                    for (int wd = 0; wd <= t >> 5; wd++) {
                        const unsigned row = s_conf[t][wd];
                        hit_acc |= (row & s_acc[wd]) != 0;
                        hit_und |= (row & s_und[wd]) != 0;
                    }
                    st = hit_acc ? 2 : hit_und ? 0 : 1;
                }
                __syncthreads();
            }
            acc = st == 1;
        }
        int rank, n_acc; // 4. output slots and the grid
        Scan(s_scan).ExclusiveSum(acc ? 1 : 0, rank, n_acc);
        if (acc && count + rank < a.max_corners) {
            const int cx = s_x[t], cy = s_y[t];
            const unsigned long long k = s_key[t];
            corners[count + rank] = make_float2((float)cx, (float)cy);
            if (scores) scores[count + rank] = __uint_as_float(~(unsigned)(k >> 32));
            if (a.suppress) grid[((cy - a.m) / a.cell) * a.gw + (cx - a.m) / a.cell] = cy * a.w + cx;
        }
        if (t == 0) s_total = min(a.max_corners, count + n_acc);
        __syncthreads(); // the grid writes and the shared arrays before the next chunk
        count = s_total;
    }
    const float nan = __int_as_float(0x7fc00000);
    for (int i = count + t; i < a.max_corners; i += SEL_CHUNK) {
        corners[i] = make_float2(nan, nan);
        if (scores) scores[i] = nan;
    }
    if (t == 0) a.counts[z] = count;
}

// Workspace of one detection call (sizes only; the caller carves it).
void plan_corners(int w, int h, int n, int win, CornerPlan *p)
{
    const int m = win / 2 + 1;
    const long long iw = (long long)w - 2 * m, ih = (long long)h - 2 * m;
    p->m = m;
    p->iw = iw > 0 ? (int)iw : 0;
    p->ih = ih > 0 ? (int)ih : 0;
    p->cap = (p->iw && p->ih) ? ((long long)(p->iw + 1) / 2) * ((p->ih + 1) / 2) : 0;
    p->total = p->cap * n;
}

// One image: a device-wide radix sort of all cap slots, the unused ones filled with ~0 (the key of score 0, which never
// qualifies, so they sort after every candidate): DeviceSegmentedSort gives a segment this large to a single CTA, which
// measured 0.48 ms for one 1080p image at window 3 against 0.071 ms here (DESIGN.md 3.6).  Several images: one segment each.
int corner_sort_bytes(long long total, int n, size_t *bytes)
{
    *bytes = 0;
    if (total == 0) return OFB_OK;
    if (n == 1)
        OFB_CUDA_TRY(cub::DeviceRadixSort::SortKeys(nullptr, *bytes, (const unsigned long long *)nullptr,
                                                    (unsigned long long *)nullptr, (int)total, 0, 64, (cudaStream_t)0));
    else
        OFB_CUDA_TRY(cub::DeviceSegmentedSort::SortKeys(nullptr, *bytes, (const unsigned long long *)nullptr,
                                                        (unsigned long long *)nullptr, (int)total, n, (int *)nullptr,
                                                        (int *)nullptr, (cudaStream_t)0));
    return OFB_OK;
}

int launch_detect_corners(const DetectArgs &d, int win, cudaStream_t st, unsigned long long *launches)
{
    const CornerPlan &p = d.plan;
    corner_init_kernel<<<(d.n + 255) / 256, 256, 0, st>>>(d.max_bits, d.seg_begin, d.seg_end, d.n, (int)p.cap);
    OFB_CUDA_TRY(cudaGetLastError());
    if (launches) ++*launches;
    CornerArgs a = {};
    a.img = d.img;
    a.pitch = d.pitch;
    a.istr = d.istr;
    a.w = d.w;
    a.h = d.h;
    a.n = d.n;
    a.m = p.m;
    a.map = d.map;
    a.map_stride = (size_t)d.w * d.h;
    a.max_bits = d.max_bits;
    int rc = launch_corner_score(a, win, st, launches);
    if (rc) return rc;
    if (p.total > 0) {
        if (d.n == 1) OFB_CUDA_TRY(cudaMemsetAsync(d.keys_in, 0xff, (size_t)p.total * sizeof(unsigned long long), st));
        const dim3 grid((unsigned)((p.iw + 31) / 32), (unsigned)min((p.ih + 7) / 8, 65535), (unsigned)d.n);
        corner_cand_kernel<<<grid, dim3(32, 8), 0, st>>>(d.map, a.map_stride, d.w, d.h, p.m, d.max_bits, d.quality_level,
                                                          d.min_score, d.seg_end, d.keys_in);
        OFB_CUDA_TRY(cudaGetLastError());
        if (launches) ++*launches;
        size_t bytes = d.sort_bytes;
        if (d.n == 1)
            OFB_CUDA_TRY(cub::DeviceRadixSort::SortKeys(d.sort_tmp, bytes, d.keys_in, d.keys_out, (int)p.total, 0, 64, st));
        else
            OFB_CUDA_TRY(cub::DeviceSegmentedSort::SortKeys(d.sort_tmp, bytes, d.keys_in, d.keys_out, (int)p.total, d.n,
                                                            d.seg_begin, d.seg_end, st));
    }
    SelArgs s = {};
    s.keys = d.keys_out;
    s.seg_begin = d.seg_begin;
    s.seg_end = d.seg_end;
    s.w = d.w;
    s.m = p.m;
    s.max_corners = d.max_corners;
    s.md2 = (double)d.min_distance * (double)d.min_distance;
    s.suppress = s.md2 > 1.0 && p.total > 0;
    if (s.suppress) {
        int c = (int)fmin(floor((double)d.min_distance / sqrt(2.0)), (double)(1 << 30));
        if (c < 1) c = 1;
        while (c > 1 && 2.0 * (double)(c - 1) * (double)(c - 1) >= s.md2) c--; // a cell never holds two accepted corners
        s.cell = c;
        s.gw = (p.iw + c - 1) / c;
        s.gh = (p.ih + c - 1) / c;
        s.reach = (int)fmin(ceil((double)d.min_distance), (double)(p.iw > p.ih ? p.iw : p.ih));
        s.grid = d.grid;
        OFB_CUDA_TRY(cudaMemsetAsync(d.grid, 0xff, (size_t)s.gw * s.gh * d.n * sizeof(int), st));
    }
    s.corners = d.corners;
    s.scores = d.scores;
    s.counts = d.counts;
    corner_select_kernel<<<d.n, SEL_CHUNK, 0, st>>>(s);
    OFB_CUDA_TRY(cudaGetLastError());
    if (launches) ++*launches;
    return OFB_OK;
}

} // namespace ofb
