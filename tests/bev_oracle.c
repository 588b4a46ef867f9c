/*
 * bev_oracle.c -- brute-force restatement of ok_bev_query's pixel classes (TEST INFRASTRUCTURE ONLY).
 *
 * Exactly the definition in include/openkitchen_b200.h: the even-odd (PNPOLY) rule over every edge (i, j = i - 1 cyclic)
 * of the four closed loops LI, LO, RI, RO, binary32, every operation rounded in the written order (compiled with
 * -ffp-contract=off).  No band table, no early exit, no margin: the GPU tests compare the kernel with this bit for bit.
 * The caller passes sin / cos of the heading, computed by the oracle's sincosf restatement (tests/bev_oracle.py).
 */
#include <stddef.h>
#include <stdint.h>

/* even-odd rule over the closed loop p[n] (interleaved xy) */
static int inside(const float *p, int n, float px, float py)
{
    int c = 0;
    for (int i = 0, j = n - 1; i < n; j = i++) {
        const float xi = p[2 * i], yi = p[2 * i + 1], xj = p[2 * j], yj = p[2 * j + 1];
        if (((yi > py) != (yj > py)) && (px < ((xj - xi) * (py - yi)) / (yj - yi) + xi))
            c = !c;
    }
    return c;
}

/* one H x W image at pose (x, y) with heading sin / cos (rs, rc): out[r * W + c] = 0 off, 1 wall, 2 lane */
void bev_oracle(const float *li, const float *lo, const float *ri, const float *ro, int n, float x, float y, float rs,
                float rc, int H, int W, float scale, float ahead, uint8_t *out)
{
    const float hc = 0.5f * (float)(H - 1), wc = 0.5f * (float)(W - 1);
#pragma omp parallel for schedule(dynamic, 1)
    for (int r = 0; r < H; ++r)
        for (int c = 0; c < W; ++c) {
            const float f  = (hc - (float)r) * scale + ahead;
            const float l  = ((float)c - wc) * scale;
            const float px = x + (f * rc - l * rs);
            const float py = y + (f * rs + l * rc);
            const int   k  = inside(li, n, px, py) + inside(lo, n, px, py) + inside(ri, n, px, py) + inside(ro, n, px, py);
            out[(size_t)r * W + c] = (uint8_t)(k == 2 ? 2 : (k & 1) ? 1 : 0);
        }
}
