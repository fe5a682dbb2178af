/*
 * fb_oracle.c -- CPU restatement of the forward-backward consistency check (csrc/fb_check.cu, include/ofb200.h).
 *
 * TEST INFRASTRUCTURE ONLY: tests/test_fb_consistency.py compiles it into a temporary directory (gcc -O2 -std=c11
 * -ffp-contract=off -fno-fast-math, the flags of oracle/Makefile, so that every fma here would have to be explicit) and
 * checks the CUDA kernel against it, and it against a numpy float32 restatement.  The check has no reference counterpart
 * (Sundaram, Brox and Keutzer 2010).
 */
#include <math.h>
#include <stddef.h>
#include <stdint.h>
/* ---------------------------------------------------------------------------------------------
 * Forward-backward consistency check (no reference counterpart; Sundaram, Brox and Keutzer 2010).
 * fwd, bwd: total flow of one pair, w x h (u,v) interleaved, in flow units; s = flow_scale px per unit.
 * Per pixel (i, j), in this order:
 *   (u, v) = fwd[i][j]; u or v not finite                           -> 3 FWD_NONFINITE
 *   du = s*u, dv = s*v; !(|du| < 32768 && |dv| < 32768)             -> 2 OUTSIDE
 *   X = j*256 + rint(du*256), Y = i*256 + rint(dv*256)  (half to even, the rounding of orc_warp_u8's bilinear mode)
 *   X < 0 || X > (w-1)*256 || Y < 0 || Y > (h-1)*256                -> 2 OUTSIDE
 *   x0 = X>>8, wx = X&255, x1 = wx ? x0+1 : x0 (a zero-weight tap is never read), same for y
 *   a component of b00, b01, b10, b11 not finite                    -> 4 BWD_NONFINITE
 *   fx = wx/256, fy = wy/256 (exact); per component top = b00 + fx*(b01-b00), bot = b10 + fx*(b11-b10),
 *   b = top + fy*(bot-top); eu = s*(u+bu), ev = s*(v+bv); err2 = eu*eu + ev*ev;
 *   mag2 = (du*du + dv*dv) + ((s*bu)*(s*bu) + (s*bv)*(s*bv))
 *   isfinite(err2) && err2 <= alpha*mag2 + beta                     -> 0 CONSISTENT, else 1 INCONSISTENT
 * Every operation is a separately rounded float (-ffp-contract=off).  err2 (may be NULL): the value above for status
 * 0 / 1, NaN otherwise.
 * ------------------------------------------------------------------------------------------- */
void orc_fb_check(const float *fwd, const float *bwd, int w, int h, float flow_scale, float alpha, float beta, float *err2,
                  uint8_t *status)
{
    const float s = flow_scale;
    for (int i = 0; i < h; i++)
        for (int j = 0; j < w; j++) {
            const size_t o = (size_t)i * w + j;
            const float u = fwd[2 * o], v = fwd[2 * o + 1];
            float e = NAN;
            uint8_t st;
            if (!isfinite(u) || !isfinite(v)) {
                st = 3;
            } else {
                const float du = s * u, dv = s * v;
                if (!(fabsf(du) < 32768.0f && fabsf(dv) < 32768.0f)) {
                    st = 2;
                } else {
                    const int X = j * 256 + (int)rintf(du * 256.0f), Y = i * 256 + (int)rintf(dv * 256.0f);
                    if (X < 0 || X > (w - 1) * 256 || Y < 0 || Y > (h - 1) * 256) {
                        st = 2;
                    } else {
                        const int x0 = X >> 8, y0 = Y >> 8, wx = X & 255, wy = Y & 255;
                        const int x1 = wx ? x0 + 1 : x0, y1 = wy ? y0 + 1 : y0;
                        const float *b00 = bwd + 2 * ((size_t)y0 * w + x0), *b01 = bwd + 2 * ((size_t)y0 * w + x1);
                        const float *b10 = bwd + 2 * ((size_t)y1 * w + x0), *b11 = bwd + 2 * ((size_t)y1 * w + x1);
                        int finite = 1;
                        for (int c = 0; c < 2; c++)
                            finite &= isfinite(b00[c]) && isfinite(b01[c]) && isfinite(b10[c]) && isfinite(b11[c]);
                        if (!finite) {
                            st = 4;
                        } else {
                            const float fx = (float)wx * (1.0f / 256.0f), fy = (float)wy * (1.0f / 256.0f);
                            float b[2];
                            for (int c = 0; c < 2; c++) {
                                const float top = b00[c] + fx * (b01[c] - b00[c]);
                                const float bot = b10[c] + fx * (b11[c] - b10[c]);
                                b[c] = top + fy * (bot - top);
                            }
                            const float eu = s * (u + b[0]), ev = s * (v + b[1]);
                            e = eu * eu + ev * ev;
                            const float sbu = s * b[0], sbv = s * b[1];
                            const float mag2 = (du * du + dv * dv) + (sbu * sbu + sbv * sbv);
                            st = (isfinite(e) && e <= alpha * mag2 + beta) ? 0 : 1;
                        }
                    }
                }
            }
            status[o] = st;
            if (err2) err2[o] = e;
        }
}
