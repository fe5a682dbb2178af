/*
 * track_oracle.c -- CPU restatement of the sparse pyramidal Lucas-Kanade tracker (csrc/track.cu, include/ofb200.h
 * ofb_track_points_device).
 *
 * TEST INFRASTRUCTURE ONLY: tests/test_track_points.py compiles it into a temporary directory (gcc -O2 -std=c11
 * -ffp-contract=off -fno-fast-math, the flags of oracle/Makefile, so that every fma here is explicit) and checks the
 * CUDA kernel against it.  The pyramid levels come from the pinned oracle (oracle.gauss_pyramid); the 2x2 solve is
 * lk_oracle.c's orc_solve_one, the reference's double-precision operation order.  The tracker has no reference
 * counterpart.
 */
#include <math.h>
#include <stddef.h>
#include <stdint.h>

#define PT_TRACKED 0
#define PT_NONFINITE 1
#define PT_LOW_TEXTURE 2
#define PT_OUTSIDE 3

/* One level: w x h u8, tightly packed. */
typedef struct {
    const uint8_t *img;
    int w, h;
} Level;

static int px(const Level *L, int x, int y) { return (x >= 0 && x < L->w && y >= 0 && y < L->h) ? L->img[(size_t)y * L->w + x] : 0; }

/* The fields of include/ofb200.h at integer position (x, y): 0 = Ix (Dx), 1 = Iy (Dy), 2 = Dt; 0 outside the level. */
static const int MASK[3][9] = {{-1, 0, 1, -2, 0, 2, -1, 0, 1}, {-1, -2, -1, 0, 0, 0, 1, 2, 1}, {1, 2, 1, 2, 3, 2, 1, 2, 1}};
static int field(const Level *L, int f, int x, int y)
{
    if (x < 0 || x >= L->w || y < 0 || y >= L->h) return 0;
    int s = 0;
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) s += MASK[f][3 * i + j] * px(L, x - 1 + j, y - 1 + i);
    return s;
}

/* 8.8 fixed-point bilinear sample at (X, Y) in 1/256 px */
static int sample(const Level *L, int f, int X, int Y)
{
    const int x0 = X >> 8, y0 = Y >> 8, wx = X & 255, wy = Y & 255;
    const int f00 = field(L, f, x0, y0), f01 = field(L, f, x0 + 1, y0);
    const int f10 = field(L, f, x0, y0 + 1), f11 = field(L, f, x0 + 1, y0 + 1);
    return ((256 - wy) * ((256 - wx) * f00 + wx * f01) + wy * ((256 - wx) * f10 + wx * f11) + 32768) >> 16;
}

/* lk_oracle.c's orc_solve_one (OptFlowGpu.cu:1829-1842 as nvcc contracts it) */
static void solve(double a, double b, double d, double sxt, double syt, float *u, float *v)
{
    const double bb = b * b;
    const double det = fma(a, d, -bb);
    const double prefix = 1.0 / det;
    const double ap = a * prefix, bp = b * prefix, dp = d * prefix;
    *u = (float)fma(bp, syt, -(dp * sxt));
    *v = (float)fma(bp, sxt, -(ap * syt));
}

static int in_range(float fs, float u, float v) { return fabsf(fs * u) < 32768.0f && fabsf(fs * v) < 32768.0f; }

/* One point: the rule of include/ofb200.h.  prev / next: levels 0..levels-1. */
static uint8_t track_one(const Level *prev, const Level *next, int levels, int win, float fs, float x, float y, int iters, float eps,
                         float min_eig, float *out)
{
    const int R = win / 2;
    const int w = prev[0].w, h = prev[0].h;
    if (!isfinite(x) || !isfinite(y) || !(x >= 0.0f && x <= (float)(w - 1) && y >= 0.0f && y <= (float)(h - 1))) {
        out[0] = out[1] = NAN;
        return PT_OUTSIDE;
    }
    const float s256 = fs * 256.0f;
    float du = 0.0f, dv = 0.0f;
    int gx[19 * 19], gy[19 * 19], sp[19 * 19];
    for (int k = levels - 1; k >= 0; k--) {
        const Level *P = &prev[k], *N = &next[k];
        const float sc = (float)(256 >> k);
        const int PX = (int)rintf(x * sc), PY = (int)rintf(y * sc);
        int a = 0, dd = 0, b = 0;
        for (int oy = -R; oy <= R; oy++)
            for (int ox = -R; ox <= R; ox++) {
                const int i = (oy + R) * win + (ox + R), X = PX + 256 * ox, Y = PY + 256 * oy;
                gx[i] = sample(P, 0, X, Y);
                gy[i] = sample(P, 1, X, Y);
                sp[i] = sample(P, 2, X, Y);
                a += gx[i] * gx[i];
                dd += gy[i] * gy[i];
                b += gx[i] * gy[i];
            }
        if (min_eig > 0.0f) {
            const double S = (double)a + (double)dd, mu = (double)min_eig * (double)(win * win);
            const double det = (double)((int64_t)a * dd - (int64_t)b * b);
            if (mu > 0.5 * S || det < mu * (S - mu)) {
                out[0] = du * (float)(1 << k);
                out[1] = dv * (float)(1 << k);
                return PT_LOW_TEXTURE;
            }
        }
        for (int it = 0; it < iters; it++) {
            if (!in_range(fs, du, dv)) {
                out[0] = du * (float)(1 << k);
                out[1] = dv * (float)(1 << k);
                return PT_OUTSIDE;
            }
            const int U = (int)rintf(du * s256), V = (int)rintf(dv * s256);
            int tx = 0, ty = 0;
            for (int oy = -R; oy <= R; oy++)
                for (int ox = -R; ox <= R; ox++) {
                    const int i = (oy + R) * win + (ox + R);
                    const int It = sample(N, 2, PX + U + 256 * ox, PY + V + 256 * oy) - sp[i];
                    tx += gx[i] * It;
                    ty += gy[i] * It;
                }
            float eu, ev;
            solve((double)a, (double)b, (double)dd, (double)tx, (double)ty, &eu, &ev);
            du += eu;
            dv += ev;
            if (!isfinite(eu) || !isfinite(ev)) {
                out[0] = du * (float)(1 << k);
                out[1] = dv * (float)(1 << k);
                return PT_NONFINITE;
            }
            if (eps > 0.0f && fabsf(fs * eu) < eps && fabsf(fs * ev) < eps) break;
        }
        if (k > 0) {
            du *= 2.0f;
            dv *= 2.0f;
        } else {
            out[0] = du;
            out[1] = dv;
            if (!in_range(fs, du, dv)) return PT_OUTSIDE;
            const int TX = PX + (int)rintf(du * s256), TY = PY + (int)rintf(dv * s256);
            if (TX < 0 || TX > (w - 1) * 256 || TY < 0 || TY > (h - 1) * 256) return PT_OUTSIDE;
        }
    }
    return PT_TRACKED;
}

/* prev_levels / next_levels: `levels` pointers to tightly packed (w>>k) x (h>>k) u8 images; points / flow: n (x, y) /
 * (u, v) float pairs; status: n bytes. */
void orc_track_points(const uint8_t *const *prev_levels, const uint8_t *const *next_levels, int w, int h, int levels, int win,
                      float flow_scale, const float *points, int n, int iters, float eps, float min_eig, float *flow,
                      uint8_t *status)
{
    Level P[8], N[8];
    for (int k = 0; k < levels; k++) {
        P[k] = (Level){prev_levels[k], w >> k, h >> k};
        N[k] = (Level){next_levels[k], w >> k, h >> k};
    }
    for (int i = 0; i < n; i++)
        status[i] = track_one(P, N, levels, win, flow_scale, points[2 * i], points[2 * i + 1], iters, eps, min_eig, flow + 2 * i);
}
