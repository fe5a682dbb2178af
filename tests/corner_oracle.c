/*
 * corner_oracle.c -- CPU restatement of the Shi-Tomasi corner detector (csrc/corners.cu, include/ofb200.h
 * ofb_min_eig_map_device / ofb_detect_corners_device).
 *
 * TEST INFRASTRUCTURE ONLY: tests/test_corners.py compiles it into a temporary directory (gcc -O2 -std=c11
 * -ffp-contract=off -fno-fast-math, the flags of track_oracle.c, so that no fma is formed) and checks the CUDA kernels
 * against it.  It is written from the rule, not from the kernels: direct window sums, qsort of the candidates, and a
 * bucket grid of side ceil(min_distance) for the greedy selection.
 */
#include <math.h>
#include <stddef.h>
#include <stdint.h>
#include <stdlib.h>

/* Sobel fields of include/ofb200.h (the tracker's Ix, Iy at level 0), 0 outside the frame. */
static int px(const uint8_t *img, size_t pitch, int w, int h, int x, int y)
{
    return (x >= 0 && x < w && y >= 0 && y < h) ? img[(size_t)y * pitch + x] : 0;
}

/* img: w x h u8 with row pitch `pitch`; score: w x h floats. */
void orc_min_eig_map(const uint8_t *img, size_t pitch, int w, int h, int win, float *score)
{
    const int R = win / 2;
    int *gx = malloc(sizeof(int) * (size_t)w * h), *gy = malloc(sizeof(int) * (size_t)w * h);
    for (int y = 0; y < h; y++)
        for (int x = 0; x < w; x++) {
#define P(dx, dy) px(img, pitch, w, h, x + (dx), y + (dy))
            gx[(size_t)y * w + x] = (P(1, -1) + 2 * P(1, 0) + P(1, 1)) - (P(-1, -1) + 2 * P(-1, 0) + P(-1, 1));
            gy[(size_t)y * w + x] = (P(-1, 1) + 2 * P(0, 1) + P(1, 1)) - (P(-1, -1) + 2 * P(0, -1) + P(1, -1));
#undef P
        }
    for (int y = 0; y < h; y++)
        for (int x = 0; x < w; x++) {
            int A = 0, D = 0, B = 0;
            for (int oy = -R; oy <= R; oy++)
                for (int ox = -R; ox <= R; ox++) {
                    const int xx = x + ox, yy = y + oy;
                    if (xx < 0 || xx >= w || yy < 0 || yy >= h) continue;
                    const int a = gx[(size_t)yy * w + xx], b = gy[(size_t)yy * w + xx];
                    A += a * a;
                    D += b * b;
                    B += a * b;
                }
            const int S = A + D;
            double l1 = 0.0;
            if (S != 0) {
                const int64_t det = (int64_t)A * D - (int64_t)B * B, T = (int64_t)A - D;
                const int64_t disc = T * T + 4 * (int64_t)B * B;
                l1 = (2.0 * (double)det) / ((double)S + sqrt((double)disc));
            }
            score[(size_t)y * w + x] = (float)(l1 / (double)(win * win));
        }
    free(gx);
    free(gy);
}

static int cmp_key(const void *a, const void *b)
{
    const uint64_t x = *(const uint64_t *)a, y = *(const uint64_t *)b;
    return x < y ? -1 : x > y;
}

static uint32_t bits(float f)
{
    union {
        float f;
        uint32_t u;
    } v = {f};
    return v.u;
}

/* score: w x h (any map, e.g. crafted); corners: max_corners (x, y) pairs; scores: max_corners or NULL.  Returns the count. */
int orc_detect_corners(const float *score, int w, int h, int win, int max_corners, float quality_level, float min_distance,
                       float min_score, float *corners, float *scores)
{
    const int m = win / 2 + 1;
    int count = 0;
    for (int k = 0; k < max_corners; k++) {
        corners[2 * k] = corners[2 * k + 1] = NAN;
        if (scores) scores[k] = NAN;
    }
    if (w < 2 * m + 1 || h < 2 * m + 1) return 0;
    float mx = 0.0f;
    for (int y = m; y <= h - 1 - m; y++)
        for (int x = m; x <= w - 1 - m; x++)
            if (score[(size_t)y * w + x] > mx) mx = score[(size_t)y * w + x];
    const float q = quality_level * mx;
    const float thr = q > min_score ? q : min_score;
    uint64_t *keys = malloc(sizeof(uint64_t) * ((size_t)(w - 2 * m) * (h - 2 * m) + 1));
    size_t nk = 0;
    for (int y = m; y <= h - 1 - m; y++)
        for (int x = m; x <= w - 1 - m; x++) {
            const float s = score[(size_t)y * w + x];
            if (!(s > thr)) continue;
            int ok = 1;
            for (int dy = -1; dy <= 1 && ok; dy++)
                for (int dx = -1; dx <= 1; dx++) {
                    const int nx = x + dx, ny = y + dy;
                    if ((dx == 0 && dy == 0) || nx < m || nx > w - 1 - m || ny < m || ny > h - 1 - m) continue;
                    const float t = score[(size_t)ny * w + nx];
                    const long pi = (long)y * w + x, qi = (long)ny * w + nx;
                    if (!(s > t || (s == t && pi < qi))) {
                        ok = 0;
                        break;
                    }
                }
            if (ok) keys[nk++] = ((uint64_t)(~bits(s)) << 32) | (uint32_t)((long)y * w + x);
        }
    qsort(keys, nk, sizeof(uint64_t), cmp_key);
    const double md2 = (double)min_distance * (double)min_distance;
    /* bucket grid of side cs >= min_distance: a conflicting corner lies in the 3x3 cells around; chained lists */
    const double big = (double)(w > h ? w : h) + 1.0;
    const int cs = (int)(ceil((double)min_distance) < 1.0 ? 1.0 : (ceil((double)min_distance) > big ? big : ceil((double)min_distance)));
    const int gw = (w + cs - 1) / cs, gh = (h + cs - 1) / cs;
    int *head = malloc(sizeof(int) * (size_t)gw * gh), *next = malloc(sizeof(int) * (size_t)(max_corners + 1));
    for (long i = 0; i < (long)gw * gh; i++) head[i] = -1;
    for (size_t i = 0; i < nk && count < max_corners; i++) {
        const int idx = (int)(uint32_t)keys[i], x = idx % w, y = idx / w, cx = x / cs, cy = y / cs;
        int ok = 1;
        for (int gy = cy - 1; gy <= cy + 1 && ok; gy++)
            for (int gx = cx - 1; gx <= cx + 1 && ok; gx++) {
                if (gx < 0 || gx >= gw || gy < 0 || gy >= gh) continue;
                for (int e = head[gy * gw + gx]; e >= 0; e = next[e]) {
                    const int64_t dx = x - (int64_t)corners[2 * e], dy = y - (int64_t)corners[2 * e + 1];
                    if ((double)(dx * dx + dy * dy) < md2) {
                        ok = 0;
                        break;
                    }
                }
            }
        if (!ok) continue;
        corners[2 * count] = (float)x;
        corners[2 * count + 1] = (float)y;
        if (scores) {
            union {
                uint32_t u;
                float f;
            } v = {~(uint32_t)(keys[i] >> 32)};
            scores[count] = v.f;
        }
        next[count] = head[cy * gw + cx];
        head[cy * gw + cx] = count;
        count++;
    }
    free(keys);
    free(head);
    free(next);
    return count;
}
