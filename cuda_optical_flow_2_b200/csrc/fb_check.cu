// fb_check.cu -- forward-backward consistency check of two total-flow fields (no reference counterpart).
//
// Per pixel: follow the forward vector, sample the backward flow there bilinearly, and compare the two
// (Sundaram, Brox and Keutzer 2010: |f + b|^2 <= alpha (|f|^2 + |b|^2) + beta).  The arithmetic is pinned so that
// this kernel, the tests' C restatement (orc_fb_check) and a numpy float32 one agree bit for bit: every multiply
// and add is rounded on its own (__fmul_rn / __fadd_rn / __fsub_rn: nvcc may not contract them into fma), and the
// displacement is rounded to 1/256 px exactly as the bilinear warp does (lk_level.cuh, __float2int_rn).
//
// Memory bound gather: 8 B of fwd (128-bit streaming loads, two pixels each), the four bwd taps through L1
// (ld.global.nc: neighbouring pixels share taps), 1 B of status (four pixels per 32-bit store) and optionally 4 B of
// err2 (float4 stores).  A thread owns four consecutive pixels of a row; rows whose addresses are not aligned for the
// wide accesses (odd widths) take the per-pixel path.
#include "ofb_common.cuh"

namespace ofb {

constexpr int FB_NT = 256; // threads per block
constexpr int FB_PX = 4;   // pixels per thread

static __device__ __forceinline__ bool fb_finite2(float2 b) { return isfinite(b.x) && isfinite(b.y); }

// One pixel (i, j) of a pair; bw is the pair's backward flow, row y at bw + y * w.  Returns the status, *err2 its squared
// error (NaN where the status is neither CONSISTENT nor INCONSISTENT).  STRIP (row strips): only backward rows [b0, b1)
// are held; a pixel that would read a tap of non-zero weight outside them is OFB_FB_UNCHECKED.  The whole-frame form
// compiles without that test.
template <bool STRIP>
static __device__ __forceinline__ uint32_t fb_pixel(float u, float v, int i, int j, const float2 *__restrict__ bw, int w,
                                                    int h, float s, float alpha, float beta, float *err2, int b0 = 0, int b1 = 0)
{
    *err2 = __int_as_float(0x7fc00000);
    if (!isfinite(u) || !isfinite(v)) return OFB_FB_FWD_NONFINITE;
    const float du = __fmul_rn(s, u), dv = __fmul_rn(s, v);
    if (!(fabsf(du) < 32768.0f && fabsf(dv) < 32768.0f)) return OFB_FB_OUTSIDE;
    const int X = j * 256 + __float2int_rn(__fmul_rn(du, 256.0f)), Y = i * 256 + __float2int_rn(__fmul_rn(dv, 256.0f));
    if (X < 0 || X > (w - 1) * 256 || Y < 0 || Y > (h - 1) * 256) return OFB_FB_OUTSIDE;
    const int x0 = X >> 8, y0 = Y >> 8, wx = X & 255, wy = Y & 255;
    const int x1 = wx ? x0 + 1 : x0, y1 = wy ? y0 + 1 : y0; // a zero-weight tap is never read
    if (STRIP && (y0 < b0 || y1 >= b1)) return OFB_FB_UNCHECKED;
    const float2 b00 = __ldg(bw + (size_t)y0 * w + x0), b01 = __ldg(bw + (size_t)y0 * w + x1);
    const float2 b10 = __ldg(bw + (size_t)y1 * w + x0), b11 = __ldg(bw + (size_t)y1 * w + x1);
    if (!(fb_finite2(b00) && fb_finite2(b01) && fb_finite2(b10) && fb_finite2(b11))) return OFB_FB_BWD_NONFINITE;
    const float fx = __fmul_rn((float)wx, 1.0f / 256.0f), fy = __fmul_rn((float)wy, 1.0f / 256.0f);
    const float tu = __fadd_rn(b00.x, __fmul_rn(fx, __fsub_rn(b01.x, b00.x)));
    const float bu_ = __fadd_rn(b10.x, __fmul_rn(fx, __fsub_rn(b11.x, b10.x)));
    const float bu = __fadd_rn(tu, __fmul_rn(fy, __fsub_rn(bu_, tu)));
    const float tv = __fadd_rn(b00.y, __fmul_rn(fx, __fsub_rn(b01.y, b00.y)));
    const float bv_ = __fadd_rn(b10.y, __fmul_rn(fx, __fsub_rn(b11.y, b10.y)));
    const float bv = __fadd_rn(tv, __fmul_rn(fy, __fsub_rn(bv_, tv)));
    const float eu = __fmul_rn(s, __fadd_rn(u, bu)), ev = __fmul_rn(s, __fadd_rn(v, bv));
    const float e2 = __fadd_rn(__fmul_rn(eu, eu), __fmul_rn(ev, ev));
    const float sbu = __fmul_rn(s, bu), sbv = __fmul_rn(s, bv);
    const float mag2 = __fadd_rn(__fadd_rn(__fmul_rn(du, du), __fmul_rn(dv, dv)), __fadd_rn(__fmul_rn(sbu, sbu), __fmul_rn(sbv, sbv)));
    *err2 = e2;
    return isfinite(e2) && e2 <= __fadd_rn(__fmul_rn(alpha, mag2), beta) ? OFB_FB_CONSISTENT : OFB_FB_INCONSISTENT;
}

// grid = (ceil(h * ceil(w / 4) / FB_NT), 1, n_pairs); thread t of a pair owns row t / ceil(w/4), columns 4 * (t % ceil(w/4)) + 0..3
template <bool ERR2>
__global__ void __launch_bounds__(FB_NT)
fb_check_kernel(const float2 *__restrict__ fwd, const float2 *__restrict__ bwd, int w, int h, int chunks, float s, float alpha,
                float beta, uint8_t *__restrict__ status, float *__restrict__ err2)
{
    const int t = blockIdx.x * FB_NT + threadIdx.x;
    if (t >= h * chunks) return;
    const int i = t / chunks, j0 = (t - i * chunks) * FB_PX;
    const size_t plane = (size_t)w * h, o = (size_t)blockIdx.z * plane + (size_t)i * w + j0;
    const float2 *bw = bwd + (size_t)blockIdx.z * plane;
    const uintptr_t al = (reinterpret_cast<uintptr_t>(fwd + o) & 15) | (reinterpret_cast<uintptr_t>(status + o) & 3) |
                         (ERR2 ? reinterpret_cast<uintptr_t>(err2 + o) & 15 : 0);
    if (j0 + FB_PX <= w && !al) {
        const float4 f01 = __ldcs(reinterpret_cast<const float4 *>(fwd + o));
        const float4 f23 = __ldcs(reinterpret_cast<const float4 *>(fwd + o) + 1);
        float4 e;
        uint32_t st = fb_pixel<false>(f01.x, f01.y, i, j0, bw, w, h, s, alpha, beta, &e.x);
        st |= fb_pixel<false>(f01.z, f01.w, i, j0 + 1, bw, w, h, s, alpha, beta, &e.y) << 8;
        st |= fb_pixel<false>(f23.x, f23.y, i, j0 + 2, bw, w, h, s, alpha, beta, &e.z) << 16;
        st |= fb_pixel<false>(f23.z, f23.w, i, j0 + 3, bw, w, h, s, alpha, beta, &e.w) << 24;
        __stcs(reinterpret_cast<unsigned *>(status + o), st);
        if (ERR2) __stcs(reinterpret_cast<float4 *>(err2 + o), e);
        return;
    }
    for (int k = 0; k < FB_PX && j0 + k < w; k++) {
        const float2 f = __ldcs(fwd + o + k);
        float e;
        status[o + k] = (uint8_t)fb_pixel<false>(f.x, f.y, i, j0 + k, bw, w, h, s, alpha, beta, &e);
        if (ERR2) err2[o + k] = e;
    }
}

// Row strips: the own rows [y0, y0 + rows) of one pair, of a frame h rows high.  fwd / status / err2 hold those rows
// only; bwd_rows holds backward rows [b0, b1).  UNCHECKED pixels set bit 2 of *flag.
// grid = ceil(rows * ceil(w / 4) / FB_NT); thread t owns local row t / ceil(w/4), columns 4 * (t % ceil(w/4)) + 0..3
template <bool ERR2>
__global__ void __launch_bounds__(FB_NT)
fb_check_strip_kernel(const float2 *__restrict__ fwd, const float2 *__restrict__ bwd_rows, int w, int h, int y0, int rows, int b0,
                      int b1, int chunks, float s, float alpha, float beta, uint8_t *__restrict__ status, float *__restrict__ err2,
                      int *__restrict__ flag)
{
    const int t = blockIdx.x * FB_NT + threadIdx.x;
    if (t >= rows * chunks) return;
    const int r = t / chunks, j0 = (t - r * chunks) * FB_PX, i = y0 + r;
    const size_t o = (size_t)r * w + j0;
    const float2 *bw = bwd_rows - (ptrdiff_t)b0 * w; // global row y at bw + y * w; only rows [b0, b1) are read
    uint32_t unchecked = 0;
    const uintptr_t al = (reinterpret_cast<uintptr_t>(fwd + o) & 15) | (reinterpret_cast<uintptr_t>(status + o) & 3) |
                         (ERR2 ? reinterpret_cast<uintptr_t>(err2 + o) & 15 : 0);
    if (j0 + FB_PX <= w && !al) {
        const float4 f01 = __ldcs(reinterpret_cast<const float4 *>(fwd + o));
        const float4 f23 = __ldcs(reinterpret_cast<const float4 *>(fwd + o) + 1);
        float4 e;
        uint32_t st = fb_pixel<true>(f01.x, f01.y, i, j0, bw, w, h, s, alpha, beta, &e.x, b0, b1);
        st |= fb_pixel<true>(f01.z, f01.w, i, j0 + 1, bw, w, h, s, alpha, beta, &e.y, b0, b1) << 8;
        st |= fb_pixel<true>(f23.x, f23.y, i, j0 + 2, bw, w, h, s, alpha, beta, &e.z, b0, b1) << 16;
        st |= fb_pixel<true>(f23.z, f23.w, i, j0 + 3, bw, w, h, s, alpha, beta, &e.w, b0, b1) << 24;
        __stcs(reinterpret_cast<unsigned *>(status + o), st);
        if (ERR2) __stcs(reinterpret_cast<float4 *>(err2 + o), e);
#pragma unroll
        for (int k = 0; k < FB_PX; k++) unchecked |= ((st >> (8 * k)) & 255u) == OFB_FB_UNCHECKED;
    } else {
        for (int k = 0; k < FB_PX && j0 + k < w; k++) {
            const float2 f = __ldcs(fwd + o + k);
            float e;
            const uint32_t st = fb_pixel<true>(f.x, f.y, i, j0 + k, bw, w, h, s, alpha, beta, &e, b0, b1);
            status[o + k] = (uint8_t)st;
            if (ERR2) err2[o + k] = e;
            unchecked |= st == OFB_FB_UNCHECKED;
        }
    }
    if (unchecked) atomicOr(flag, 4);
}

int launch_fb_check_strip(const float *fwd, const float *bwd_rows, int w, int h, int y0, int rows, int b0, int b1, float flow_scale,
                          float alpha, float beta, uint8_t *status, float *err2, int *flag, cudaStream_t stream,
                          unsigned long long *launches)
{
    if (w < 1 || h < 1 || w > 32768 || h > 32768 || rows < 1 || y0 < 0 || y0 + rows > h || b0 > y0 || b1 < y0 + rows) {
        set_error("fb_check_strip: bad geometry (w %d h %d rows [%d,%d) held [%d,%d))", w, h, y0, y0 + rows, b0, b1);
        return OFB_ERR_INVALID;
    }
    const int chunks = (w + FB_PX - 1) / FB_PX;
    const long long threads = (long long)rows * chunks;
    const unsigned grid = (unsigned)((threads + FB_NT - 1) / FB_NT);
    const float2 *f = reinterpret_cast<const float2 *>(fwd), *b = reinterpret_cast<const float2 *>(bwd_rows);
    if (err2)
        fb_check_strip_kernel<true><<<grid, FB_NT, 0, stream>>>(f, b, w, h, y0, rows, b0, b1, chunks, flow_scale, alpha, beta, status,
                                                               err2, flag);
    else
        fb_check_strip_kernel<false><<<grid, FB_NT, 0, stream>>>(f, b, w, h, y0, rows, b0, b1, chunks, flow_scale, alpha, beta, status,
                                                                nullptr, flag);
    OFB_CUDA_TRY(cudaGetLastError());
    if (launches) ++*launches;
    return OFB_OK;
}

int preload_fb_check_strip()
{
    cudaFuncAttributes fa;
    OFB_CUDA_TRY(cudaFuncGetAttributes(&fa, fb_check_strip_kernel<true>));
    OFB_CUDA_TRY(cudaFuncGetAttributes(&fa, fb_check_strip_kernel<false>));
    return OFB_OK;
}

int launch_fb_check(const float *fwd, const float *bwd, int w, int h, int n_pairs, float flow_scale, float alpha, float beta,
                    uint8_t *status, float *err2, cudaStream_t stream, unsigned long long *launches)
{
    if (w < 1 || h < 1 || w > 32768 || h > 32768 || n_pairs < 1 || n_pairs > 65535) {
        set_error("fb_check: bad geometry (w %d h %d pairs %d; at most 32768 x 32768 pixels and 65535 pairs)", w, h, n_pairs);
        return OFB_ERR_INVALID;
    }
    const int chunks = (w + FB_PX - 1) / FB_PX;
    const long long threads = (long long)h * chunks;
    const dim3 grid((unsigned)((threads + FB_NT - 1) / FB_NT), 1, (unsigned)n_pairs);
    const float2 *f = reinterpret_cast<const float2 *>(fwd), *b = reinterpret_cast<const float2 *>(bwd);
    if (err2) fb_check_kernel<true><<<grid, FB_NT, 0, stream>>>(f, b, w, h, chunks, flow_scale, alpha, beta, status, err2);
    else fb_check_kernel<false><<<grid, FB_NT, 0, stream>>>(f, b, w, h, chunks, flow_scale, alpha, beta, status, nullptr);
    OFB_CUDA_TRY(cudaGetLastError());
    if (launches) ++*launches;
    return OFB_OK;
}

} // namespace ofb
