// track.cu -- sparse pyramidal Lucas-Kanade: a list of sub-pixel points followed through the pyramid, iterated per
// level (the KLT tracker; no reference counterpart).  The rule is pinned in include/ofb200.h (ofb_track_points_device):
// 8.8 fixed-point positions, the reference's derivative masks as exact integer fields, the warp's bilinear rule on those
// fields, exact int32 window sums and the reference's double-precision 2x2 solve (lk_solve1), so that this kernel and
// the tests' C restatement (tests/track_oracle.c) agree bit for bit.
//
// One warp per point, one launch for every level: the pyramids are complete before the kernel starts and points are
// independent.  Per level the warp stages the (WIN+3)^2 bytes of prev_k around the point in shared memory, builds Ix, Iy
// and Sp = Dt (*) prev_k on the (WIN+1)^2 integer positions the samples' taps touch, samples the three fields at the WIN^2
// window positions (each lane keeps its samples in registers for the whole level) and reduces the three tensor sums
// across the warp.  Per iteration it stages the bytes of next_k around the target, builds Sn = Dt (*) next_k, samples it,
// reduces the two mismatch sums and solves.  Every lane holds the reduced sums and runs the same solve (SIMT: one lane
// would take the same issue slots), so no broadcast is needed.  Loads are plain ld.global.nc: the access is scattered and
// latency bound, and neighbouring points share lines through L1.
#include "lk_level.cuh"

#include <cmath>

namespace ofb {

constexpr int TRK_WARPS = 4; // points per CTA; registers held to 4 CTAs per SM (<= 128: without the bound ptxas spills
                              // at windows 7 and 9 and takes 168 at 17 and 19)

template <int WIN> struct TrkCfg {
    static constexpr int R = WIN / 2;
    static constexpr int P = WIN + 3;                 // staged image patch, P x P bytes
    static constexpr int G = WIN + 1;                 // field grid, G x G
    static constexpr int NP = (P * P + 31) / 32;      // patch bytes per lane
    static constexpr int NG = (G * G + 31) / 32;      // grid values per lane
    static constexpr int NS = (WIN * WIN + 31) / 32;  // window samples per lane
    static constexpr int PB = (P * P + 15) / 16 * 16; // patch bytes, padded
};

// The P x P bytes of one level image whose top-left is image pixel (x0, y0); 0 outside the level.
template <int WIN>
__device__ __forceinline__ void trk_stage(const uint8_t *__restrict__ img, size_t pitch, int w, int h, int x0, int y0,
                                          uint8_t *patch, int lane)
{
    using C = TrkCfg<WIN>;
#pragma unroll
    for (int j = 0; j < C::NP; j++) {
        const int t = lane + 32 * j;
        if (t < C::P * C::P) {
            const int r = t / C::P, c = t - r * C::P, y = y0 + r, x = x0 + c;
            patch[t] = (x >= 0 && x < w && y >= 0 && y < h) ? __ldg(img + (size_t)y * pitch + x) : (uint8_t)0;
        }
    }
}

// 8.8 bilinear of the grid g at tap (gi = row * G + col) with weights wx, wy (include/ofb200.h)
template <int G>
__device__ __forceinline__ int trk_bilerp(const int *g, int gi, int wx, int wy)
{
    const int ix = 256 - wx, iy = 256 - wy;
    return (iy * (ix * g[gi] + wx * g[gi + 1]) + wy * (ix * g[gi + G] + wx * g[gi + G + 1]) + 32768) >> 16;
}

template <int WIN>
__global__ void __launch_bounds__(TRK_WARPS * 32, 4) track_points_kernel(const TrackArgs a)
{
    using C = TrkCfg<WIN>;
    constexpr int R = C::R, P = C::P, G = C::G;
    __shared__ __align__(16) uint8_t s_patch[TRK_WARPS][C::PB];
    __shared__ int s_grid[TRK_WARPS][3][G * G];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int pt = blockIdx.x * TRK_WARPS + wid;
    if (pt >= a.n_points) return; // whole warps only: nothing below synchronises beyond the warp
    const size_t pair = blockIdx.z, o = pair * (size_t)a.n_points + pt;
    uint8_t *patch = s_patch[wid];
    int *gx = s_grid[wid][0], *gy = s_grid[wid][1], *gs = s_grid[wid][2];
    const float2 p0 = __ldg(reinterpret_cast<const float2 *>(a.points) + o);
    if (!(isfinite(p0.x) && isfinite(p0.y) && p0.x >= 0.0f && p0.x <= (float)(a.w - 1) && p0.y >= 0.0f &&
          p0.y <= (float)(a.h - 1))) {
        if (lane == 0) {
            reinterpret_cast<float2 *>(a.flow)[o] = make_float2(__int_as_float(0x7fc00000), __int_as_float(0x7fc00000));
            a.status[o] = OFB_PT_OUTSIDE;
        }
        return;
    }
    const float fs = a.flow_scale, s256 = __fmul_rn(a.flow_scale, 256.0f);
    const double win2 = (double)(2 * WIN * WIN);
    float2 od = make_float2(0.0f, 0.0f); // the flow reported: od at level ok, status ost
    int ok = 0, ost = OFB_PT_TRACKED;
    float2 d = make_float2(0.0f, 0.0f);
    int PX = 0, PY = 0;
    for (int k = a.levels - 1; k >= 0; k--) {
        const int wk = a.w >> k, hk = a.h >> k;
        const float sc = (float)(256 >> k); // 256 / 2^k: the products below are exact, only rint rounds
        PX = __float2int_rn(__fmul_rn(p0.x, sc));
        PY = __float2int_rn(__fmul_rn(p0.y, sc));
        const int bx = (PX >> 8) - R, by = (PY >> 8) - R, wx = PX & 255, wy = PY & 255; // grid (0, 0) = pixel (bx, by)
        // ---- prev_k: Ix, Iy, Sp on the grid, sampled at the WIN^2 window positions
        __syncwarp();
        trk_stage<WIN>(a.prev[k] + pair * a.istr[k], a.pitch[k], wk, hk, bx - 1, by - 1, patch, lane);
        __syncwarp();
#pragma unroll
        for (int j = 0; j < C::NG; j++) {
            const int t = lane + 32 * j;
            if (t < G * G) {
                const int r = t / G, c = t - r * G, x = bx + c, y = by + r;
                int ix = 0, iy = 0, sp = 0;
                if (x >= 0 && x < wk && y >= 0 && y < hk) {
                    const uint8_t *q = patch + r * P + c; // 3x3 neighbourhood, top-left
                    const int p00 = q[0], p01 = q[1], p02 = q[2], p10 = q[P], p11 = q[P + 1], p12 = q[P + 2];
                    const int p20 = q[2 * P], p21 = q[2 * P + 1], p22 = q[2 * P + 2];
                    const int top = p00 + 2 * p01 + p02, bot = p20 + 2 * p21 + p22;
                    ix = (p02 + 2 * p12 + p22) - (p00 + 2 * p10 + p20);
                    iy = bot - top;
                    sp = top + bot + 2 * (p10 + p12) + 3 * p11;
                }
                gx[t] = ix;
                gy[t] = iy;
                gs[t] = sp;
            }
        }
        __syncwarp();
        int sIx[C::NS], sIy[C::NS], sSp[C::NS];
        int sxx = 0, syy = 0, sxy = 0;
#pragma unroll
        for (int j = 0; j < C::NS; j++) {
            const int t = lane + 32 * j;
            sIx[j] = sIy[j] = sSp[j] = 0;
            if (t < WIN * WIN) {
                const int oy = t / WIN, gi = oy * G + (t - oy * WIN);
                sIx[j] = trk_bilerp<G>(gx, gi, wx, wy);
                sIy[j] = trk_bilerp<G>(gy, gi, wx, wy);
                sSp[j] = trk_bilerp<G>(gs, gi, wx, wy);
                sxx += sIx[j] * sIx[j];
                syy += sIy[j] * sIy[j];
                sxy += sIx[j] * sIy[j];
            }
        }
        sxx = __reduce_add_sync(0xffffffffu, sxx);
        syy = __reduce_add_sync(0xffffffffu, syy);
        sxy = __reduce_add_sync(0xffffffffu, sxy);
        // lam < min_eig, lam = ((A + D) - sqrt(disc)) / (2 WIN^2), as (A + D) - M < sqrt(disc) with M = 2 WIN^2 min_eig
        // (exact in double), squared: no square root and no division, whose slow paths are subroutine calls that make
        // ptxas spill around them
        if (a.min_eig > 0.0f) {
            const double A = (double)sxx, D = (double)syy, B = (double)sxy, t = __dsub_rn(A, D);
            const double disc = __dadd_rn(__dmul_rn(t, t), __dmul_rn(4.0, __dmul_rn(B, B)));
            const double T = __dsub_rn(__dadd_rn(A, D), __dmul_rn((double)a.min_eig, win2));
            if (T < 0.0 || __dmul_rn(T, T) < disc) {
                od = d, ok = k, ost = OFB_PT_LOW_TEXTURE;
                break;
            }
        }
        // ---- iterations: next_k around the target, Sn sampled, the mismatch sums, the solve
        bool stop = false;
        for (int it = 0; it < a.iters; it++) {
            if (!(fabsf(__fmul_rn(fs, d.x)) < 32768.0f && fabsf(__fmul_rn(fs, d.y)) < 32768.0f)) {
                od = d, ok = k, ost = OFB_PT_OUTSIDE;
                stop = true;
                break;
            }
            const int TX = PX + __float2int_rn(__fmul_rn(d.x, s256)), TY = PY + __float2int_rn(__fmul_rn(d.y, s256));
            const int tbx = (TX >> 8) - R, tby = (TY >> 8) - R, twx = TX & 255, twy = TY & 255;
            __syncwarp();
            trk_stage<WIN>(a.next[k] + pair * a.istr[k], a.pitch[k], wk, hk, tbx - 1, tby - 1, patch, lane);
            __syncwarp();
#pragma unroll
            for (int j = 0; j < C::NG; j++) {
                const int t = lane + 32 * j;
                if (t < G * G) {
                    const int r = t / G, c = t - r * G, x = tbx + c, y = tby + r;
                    int sn = 0;
                    if (x >= 0 && x < wk && y >= 0 && y < hk) {
                        const uint8_t *q = patch + r * P + c;
                        sn = (q[0] + 2 * q[1] + q[2]) + (q[2 * P] + 2 * q[2 * P + 1] + q[2 * P + 2]) +
                             2 * (q[P] + q[P + 2]) + 3 * q[P + 1];
                    }
                    gx[t] = sn;
                }
            }
            __syncwarp();
            int sxt = 0, syt = 0;
#pragma unroll
            for (int j = 0; j < C::NS; j++) {
                const int t = lane + 32 * j;
                if (t < WIN * WIN) {
                    const int oy = t / WIN, gi = oy * G + (t - oy * WIN);
                    const int It = trk_bilerp<G>(gx, gi, twx, twy) - sSp[j];
                    sxt += sIx[j] * It;
                    syt += sIy[j] * It;
                }
            }
            sxt = __reduce_add_sync(0xffffffffu, sxt);
            syt = __reduce_add_sync(0xffffffffu, syt);
            const float2 delta = lk_solve1(sxx, syy, sxy, sxt, syt);
            d.x = __fadd_rn(d.x, delta.x);
            d.y = __fadd_rn(d.y, delta.y);
            if (!(isfinite(delta.x) && isfinite(delta.y))) {
                od = d, ok = k, ost = OFB_PT_NONFINITE;
                stop = true;
                break;
            }
            if (a.eps > 0.0f && fabsf(__fmul_rn(fs, delta.x)) < a.eps && fabsf(__fmul_rn(fs, delta.y)) < a.eps) break;
        }
        if (stop) break;
        if (k == 0) {
            od = d;
            if (!(fabsf(__fmul_rn(fs, d.x)) < 32768.0f && fabsf(__fmul_rn(fs, d.y)) < 32768.0f)) {
                ost = OFB_PT_OUTSIDE;
            } else {
                const int TX = PX + __float2int_rn(__fmul_rn(d.x, s256)), TY = PY + __float2int_rn(__fmul_rn(d.y, s256));
                if (TX < 0 || TX > (a.w - 1) * 256 || TY < 0 || TY > (a.h - 1) * 256) ost = OFB_PT_OUTSIDE;
            }
        } else {
            d.x = __fmul_rn(d.x, 2.0f);
            d.y = __fmul_rn(d.y, 2.0f);
        }
    }
    if (lane == 0) { // (the index is formed again here rather than kept live through the level loop)
        const size_t oo = (size_t)blockIdx.z * a.n_points + pt;
        const float m = (float)(1 << ok);
        reinterpret_cast<float2 *>(a.flow)[oo] = make_float2(__fmul_rn(od.x, m), __fmul_rn(od.y, m));
        a.status[oo] = (uint8_t)ost;
    }
}

int launch_track_points(const TrackArgs &a, int win, cudaStream_t stream, unsigned long long *launches)
{
    if (a.n_points < 1 || a.n_pairs < 1 || a.n_pairs > 65535) {
        set_error("track_points: %d points x %d pairs (at most 65535 pairs)", a.n_points, a.n_pairs);
        return OFB_ERR_INVALID;
    }
    const dim3 grid((unsigned)((a.n_points + TRK_WARPS - 1) / TRK_WARPS), 1, (unsigned)a.n_pairs);
    switch (win) {
#define OFB_TRK_CASE(W)                                                              \
    case W: track_points_kernel<W><<<grid, TRK_WARPS * 32, 0, stream>>>(a); break;
        OFB_TRK_CASE(3)
        OFB_TRK_CASE(5)
        OFB_TRK_CASE(7)
        OFB_TRK_CASE(9)
        OFB_TRK_CASE(11)
        OFB_TRK_CASE(13)
        OFB_TRK_CASE(15)
        OFB_TRK_CASE(17)
        OFB_TRK_CASE(19)
#undef OFB_TRK_CASE
    default:
        set_error("track_points: window %d not supported (odd 3..%d)", win, OFB_MAX_WINDOW);
        return OFB_ERR_UNSUPPORTED;
    }
    OFB_CUDA_TRY(cudaGetLastError());
    if (launches) ++*launches;
    return OFB_OK;
}

} // namespace ofb
