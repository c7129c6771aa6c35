/*
 * recon_oracle.c -- TEST INFRASTRUCTURE (see recon_oracle.h).  Plain-C CPU
 * restatement of the reference's intra reconstruction and export path.
 * Citations are relative to /root/reference/minivideo/src/ (the reference tree
 * is not part of this repository); "spec" = ITU-T H.264.
 *
 * Differences from the reference, all outside the streams the generator emits:
 *  - Intra16x16 luma DC scaling uses the spec condition qP >= 36; the reference
 *    tests qP > 36 and executes `1 << -1` at QP'Y == 36 (h264_transform.c:797-808).
 *  - integer products, shifts and sums wrap modulo 2^32 instead of being undefined
 *    (products and shifts through wmul/wshl, sums through -fwrapv, oracle/Makefile).
 *  - a prediction mode whose neighbours are missing predicts 0 like the
 *    reference's zero-initialised block (h264_intra_prediction.c:442,:1242);
 *    neighbour values the reference would read uninitialised are taken as 0.
 */
#include "recon_oracle.h"

#include <string.h>

static inline int clip8(int v) { return v < 0 ? 0 : (v > 255 ? 255 : v); }   /* utils.c:407-415 */
static inline int32_t wmul(int32_t a, int32_t b) { return (int32_t)((uint32_t)a * (uint32_t)b); }
static inline int32_t wshl(int32_t a, int n) { return (int32_t)((uint32_t)a << n); }

/* frame zig-zag scans: zz[k] = row*n + col (utils.h:64,:74-80; spec Table 8-13/8-14) */
static uint8_t zz4[16], zz8[64];
static int zz_ready;
static void zz_build(int n, uint8_t *zz)
{
    int r = 0, c = 0, k = 0, going_up = 1;
    while (k < n * n) {
        zz[k++] = (uint8_t)(r * n + c);
        if (going_up) {
            if (c == n - 1)      { r++; going_up = 0; }
            else if (r == 0)     { c++; going_up = 0; }
            else                 { r--; c++; }
        } else {
            if (r == n - 1)      { c++; going_up = 1; }
            else if (c == 0)     { r++; going_up = 1; }
            else                 { r++; c--; }
        }
    }
}
static void zz_init(void)
{
    if (!zz_ready) { zz_build(4, zz4); zz_build(8, zz8); zz_ready = 1; }
}

/* ------------------------------------------------------------------------ */

void oracle_build_level_scale(const uint8_t *lists4x4, const uint8_t *list8x8,
                              int32_t ls4[3][6][16], int32_t ls8[6][64])
{
    /* h264.c:428-446 */
    static const int v4[6][3] = {{10,16,13},{11,18,14},{13,20,16},{14,23,18},{16,25,20},{18,29,23}};
    static const int v8[6][6] = {{20,18,32,19,25,24},{22,19,35,21,28,26},{26,23,42,24,33,31},
                                 {28,25,45,26,35,33},{32,28,51,30,40,38},{36,32,58,34,46,43}};
    zz_init();
    for (int c = 0; c < 3; c++) {
        int m[16];
        for (int k = 0; k < 16; k++) m[zz4[k]] = lists4x4 ? lists4x4[c * 16 + k] : 16;   /* h264_transform.c:440 */
        for (int q = 0; q < 6; q++)
            for (int i = 0; i < 4; i++)
                for (int j = 0; j < 4; j++) {
                    int na = (i % 2 == 0 && j % 2 == 0) ? v4[q][0] : (i % 2 == 1 && j % 2 == 1) ? v4[q][1] : v4[q][2];
                    ls4[c][q][i * 4 + j] = m[i * 4 + j] * na;                           /* h264_transform.c:675 */
                }
    }
    int m8[64];
    for (int k = 0; k < 64; k++) m8[zz8[k]] = list8x8 ? list8x8[k] : 16;
    for (int q = 0; q < 6; q++)
        for (int i = 0; i < 8; i++)
            for (int j = 0; j < 8; j++) {
                int na;                                                                   /* h264.c:471-482 */
                if (i % 4 == 0 && j % 4 == 0) na = v8[q][0];
                else if (i % 2 == 1 && j % 2 == 1) na = v8[q][1];
                else if (i % 4 == 2 && j % 4 == 2) na = v8[q][2];
                else if ((i % 4 == 0 && j % 2 == 1) || (i % 2 == 1 && j % 4 == 0)) na = v8[q][3];
                else if ((i % 4 == 0 && j % 4 == 2) || (i % 4 == 2 && j % 4 == 0)) na = v8[q][4];
                else na = v8[q][5];
                ls8[q][i * 8 + j] = m8[i * 8 + j] * na;                                   /* h264_transform.c:727 */
            }
}

int oracle_chroma_qp(int qp_y, int offset)
{
    /* h264_transform.c:71 (Table 8-15), :621-632; QpBdOffsetC == 0 (8-bit only) */
    static const int qpc_tab[22] = {29,30,31,32,32,33,34,34,35,35,36,36,37,37,37,38,38,38,39,39,39,39};
    int qpi = qp_y + offset;
    if (qpi < 0) qpi = 0;
    if (qpi > 51) qpi = 51;
    return qpi < 30 ? qpi : qpc_tab[qpi - 30];
}

/* h264_transform.c:1100-1134 (quant4x4); c,d row-major [i*4+j] */
static void scale4x4(const int32_t c[16], const int32_t ls[16], int qp, int keep_dc, int32_t d[16])
{
    int sh = qp / 6;
    for (int k = 0; k < 16; k++) {
        int32_t t = wmul(c[k], ls[k]);
        d[k] = qp > 23 ? wshl(t, sh - 4) : (int32_t)((t + (1 << (3 - sh))) >> (4 - sh));
    }
    if (keep_dc) d[0] = c[0];
}

/* h264_transform.c:1145-1191 (idct4x4), spec 8.5.12.2 */
static void inverse4x4(const int32_t d[16], int32_t r[16])
{
    int32_t f[16], h[16];
    for (int i = 0; i < 4; i++) {
        const int32_t *x = d + 4 * i;
        int32_t e0 = x[0] + x[2], e1 = x[0] - x[2], e2 = (x[1] >> 1) - x[3], e3 = x[1] + (x[3] >> 1);
        f[4 * i + 0] = e0 + e3; f[4 * i + 1] = e1 + e2; f[4 * i + 2] = e1 - e2; f[4 * i + 3] = e0 - e3;
    }
    for (int j = 0; j < 4; j++) {
        int32_t g0 = f[j] + f[8 + j], g1 = f[j] - f[8 + j];
        int32_t g2 = (f[4 + j] >> 1) - f[12 + j], g3 = f[4 + j] + (f[12 + j] >> 1);
        h[j] = g0 + g3; h[4 + j] = g1 + g2; h[8 + j] = g1 - g2; h[12 + j] = g0 - g3;
    }
    for (int k = 0; k < 16; k++) r[k] = (h[k] + 32) >> 6;
}

/* one 1-D pass of the 8x8 inverse transform, spec 8.5.13.2 / h264_transform.c:1308-1378 */
static void inverse8_1d(const int32_t in[8], int32_t out[8])
{
    int32_t a0 = in[0] + in[4];
    int32_t a1 = -in[3] + in[5] - in[7] - (in[7] >> 1);
    int32_t a2 = in[0] - in[4];
    int32_t a3 = in[1] + in[7] - in[3] - (in[3] >> 1);
    int32_t a4 = (in[2] >> 1) - in[6];
    int32_t a5 = -in[1] + in[7] + in[5] + (in[5] >> 1);
    int32_t a6 = in[2] + (in[6] >> 1);
    int32_t a7 = in[3] + in[5] + in[1] + (in[1] >> 1);
    int32_t b0 = a0 + a6, b1 = a1 + (a7 >> 2), b2 = a2 + a4, b3 = a3 + (a5 >> 2);
    int32_t b4 = a2 - a4, b5 = (a3 >> 2) - a5, b6 = a0 - a6, b7 = a7 - (a1 >> 2);
    out[0] = b0 + b7; out[1] = b2 + b5; out[2] = b4 + b3; out[3] = b6 + b1;
    out[4] = b6 - b1; out[5] = b4 - b3; out[6] = b2 - b5; out[7] = b0 - b7;
}

/* h264_transform.c:1256-1284 (quant8x8) + :1295-1383 (idct8x8) */
static void residual8x8(const int32_t c[64], const int32_t ls[64], int qp, int32_t r[64])
{
    int32_t d[64], g[64], col[8], res[8];
    int sh = qp / 6;
    for (int k = 0; k < 64; k++) {
        int32_t t = wmul(c[k], ls[k]);
        d[k] = qp > 35 ? wshl(t, sh - 6) : (int32_t)((t + (1 << (5 - sh))) >> (6 - sh));
    }
    for (int i = 0; i < 8; i++) inverse8_1d(d + 8 * i, g + 8 * i);
    for (int j = 0; j < 8; j++) {
        for (int i = 0; i < 8; i++) col[i] = g[8 * i + j];
        inverse8_1d(col, res);
        for (int i = 0; i < 8; i++) r[8 * i + j] = (res[i] + 32) >> 6;
    }
}

/* position (in samples) of 4x4 luma block blk inside its MB: h264_spatial.c:210-225 */
static inline int blk4_x(int blk) { return 4 * ((blk & 1) + 2 * ((blk >> 2) & 1)); }
static inline int blk4_y(int blk) { return 4 * (((blk >> 1) & 1) + 2 * (blk >> 3)); }

void oracle_mb_residual(const oracle_sps *sps, int mb_kind, int qp_y,
                        const int16_t coeff[384], int32_t residual[384])
{
    int32_t c[64], d[16], r[64];
    zz_init();
    const int32_t *lsY = sps->level_scale4x4[0][qp_y % 6];

    if (mb_kind == 1) {                              /* h264_transform.c:236-271 */
        for (int b8 = 0; b8 < 4; b8++) {
            for (int k = 0; k < 64; k++) c[zz8[k]] = coeff[b8 * 64 + k];
            residual8x8(c, sps->level_scale8x8[qp_y % 6], qp_y, r);
            int xo = (b8 & 1) * 8, yo = (b8 >> 1) * 8;          /* h264_spatial.c:248-260 */
            for (int i = 0; i < 8; i++)
                for (int j = 0; j < 8; j++) residual[(yo + i) * 16 + xo + j] = r[i * 8 + j];
        }
    } else {
        int32_t dcY[16];
        if (mb_kind == 2) {                          /* h264_transform.c:756-812 */
            int32_t m[16], t[16];
            for (int blk = 0; blk < 16; blk++)       /* slot 0 of blk holds c[i][j], (i,j) = blk position */
                m[(blk4_y(blk) / 4) * 4 + blk4_x(blk) / 4] = coeff[blk * 16];
            for (int j = 0; j < 4; j++) {            /* f = H * c * H, H = h264_transform.c:62-68 */
                int32_t a = m[j], b = m[4 + j], cc = m[8 + j], dd = m[12 + j];
                t[j] = a + b + cc + dd; t[4 + j] = a + b - cc - dd; t[8 + j] = a - b - cc + dd; t[12 + j] = a - b + cc - dd;
            }
            for (int i = 0; i < 4; i++) {
                int32_t a = t[4 * i], b = t[4 * i + 1], cc = t[4 * i + 2], dd = t[4 * i + 3];
                int32_t f[4] = {a + b + cc + dd, a + b - cc - dd, a - b - cc + dd, a - b + cc - dd};
                int sh = qp_y / 6;
                for (int j = 0; j < 4; j++) {
                    int32_t v = wmul(f[j], lsY[0]);
                    dcY[4 * i + j] = qp_y >= 36 ? wshl(v, sh - 6) : (int32_t)((v + (1 << (5 - sh))) >> (6 - sh));
                }
            }
        }
        for (int blk = 0; blk < 16; blk++) {         /* h264_transform.c:121-156, :184-205 */
            for (int k = 0; k < 16; k++) c[zz4[k]] = coeff[blk * 16 + k];
            if (mb_kind == 2) c[0] = dcY[(blk4_y(blk) / 4) * 4 + blk4_x(blk) / 4];
            scale4x4(c, lsY, qp_y, mb_kind == 2, d);
            inverse4x4(d, r);
            for (int i = 0; i < 4; i++)
                for (int j = 0; j < 4; j++) residual[(blk4_y(blk) + i) * 16 + blk4_x(blk) + j] = r[i * 4 + j];
        }
    }

    for (int p = 0; p < 2; p++) {                    /* h264_transform.c:286-402 */
        int qpc = oracle_chroma_qp(qp_y, p == 0 ? sps->cb_qp_offset : sps->cr_qp_offset);
        const int32_t *ls = sps->level_scale4x4[p + 1][qpc % 6];
        const int16_t *cc = coeff + 256 + p * 64;
        int32_t c00 = cc[0], c01 = cc[16], c10 = cc[32], c11 = cc[48];
        int32_t f[4] = {c00 + c01 + c10 + c11, c00 - c01 + c10 - c11,          /* :988-1005 */
                        c00 + c01 - c10 - c11, c00 - c01 - c10 + c11};
        int32_t dcC[4];
        for (int k = 0; k < 4; k++) dcC[k] = wshl(wmul(f[k], ls[0]), qpc / 6) >> 5;   /* :935 */
        for (int blk = 0; blk < 4; blk++) {
            for (int k = 0; k < 16; k++) c[zz4[k]] = cc[blk * 16 + k];
            c[0] = dcC[blk];                         /* raster_8x8_2d, utils.h:58 */
            scale4x4(c, ls, qpc, 1, d);
            inverse4x4(d, r);
            int xo = (blk & 1) * 4, yo = (blk >> 1) * 4;             /* h264_spatial.c:278-290 */
            for (int i = 0; i < 4; i++)
                for (int j = 0; j < 4; j++) residual[256 + p * 64 + (yo + i) * 8 + xo + j] = r[i * 4 + j];
        }
    }
}

/* ------------------------------------------------------------------------ */
/* Intra prediction.  pix points at the block's top-left sample in a plane.  */

#define PX(x, y) ((int)pix[(y) * stride + (x)])

/* Intra4x4 / Intra8x8 directional predictors share their formulas once the
 * neighbours are in arrays: t[x] = p[x,-1] (x = 0..2n-1), l[y] = p[-1,y],
 * tl = p[-1,-1].  n = 4: spec 8.3.1.2.x, h264_intra_prediction.c:496-926;
 * n = 8: spec 8.3.2.2.x, :1366-1793. */
static void predict_nxn(int n, int mode, const int *t, const int *l, int tl,
                        int have_left, int have_up, int have_upleft, uint8_t *pred /* [y*n+x] */)
{
    /* p(-1..) helpers over a single line: T(-1) = tl, L(-1) = tl */
#define T(i) ((i) < 0 ? tl : t[i])
#define L(i) ((i) < 0 ? tl : l[i])
    memset(pred, 0, (size_t)(n * n));
    int last = 2 * n - 1;
    switch (mode) {
    case 0: if (!have_up) return;
        for (int y = 0; y < n; y++) for (int x = 0; x < n; x++) pred[y * n + x] = (uint8_t)t[x];
        break;
    case 1: if (!have_left) return;
        for (int y = 0; y < n; y++) for (int x = 0; x < n; x++) pred[y * n + x] = (uint8_t)l[y];
        break;
    case 2: {
        int st = 0, sl = 0, v, lg = (n == 4) ? 2 : 3;
        for (int i = 0; i < n; i++) { st += t[i]; sl += l[i]; }
        if (have_left && have_up) v = (st + sl + n) >> (lg + 1);
        else if (have_left) v = (sl + n / 2) >> lg;
        else if (have_up) v = (st + n / 2) >> lg;
        else v = 128;
        memset(pred, v, (size_t)(n * n));
        break; }
    case 3: if (!have_up) return;                       /* Diagonal_Down_Left */
        for (int y = 0; y < n; y++) for (int x = 0; x < n; x++)
            pred[y * n + x] = (uint8_t)((x == n - 1 && y == n - 1)
                ? (t[last - 1] + 3 * t[last] + 2) >> 2
                : (t[x + y] + 2 * t[x + y + 1] + t[x + y + 2] + 2) >> 2);
        break;
    case 4: if (!(have_left && have_up && have_upleft)) return;   /* Diagonal_Down_Right */
        for (int y = 0; y < n; y++) for (int x = 0; x < n; x++) {
            int v;
            if (x > y) v = (T(x - y - 2) + 2 * T(x - y - 1) + T(x - y) + 2) >> 2;
            else if (x < y) v = (L(y - x - 2) + 2 * L(y - x - 1) + L(y - x) + 2) >> 2;
            else v = (t[0] + 2 * tl + l[0] + 2) >> 2;
            pred[y * n + x] = (uint8_t)v;
        }
        break;
    case 5: if (!(have_left && have_up && have_upleft)) return;   /* Vertical_Right */
        for (int y = 0; y < n; y++) for (int x = 0; x < n; x++) {
            int z = 2 * x - y, v;
            if (z >= 0 && (z & 1) == 0) v = (T(x - (y >> 1) - 1) + T(x - (y >> 1)) + 1) >> 1;
            else if (z >= 0) v = (T(x - (y >> 1) - 2) + 2 * T(x - (y >> 1) - 1) + T(x - (y >> 1)) + 2) >> 2;
            else if (z == -1) v = (l[0] + 2 * tl + t[0] + 2) >> 2;
            else if (n == 4) v = (L(y - 1) + 2 * L(y - 2) + L(y - 3) + 2) >> 2;
            else v = (L(y - 2 * x - 1) + 2 * L(y - 2 * x - 2) + L(y - 2 * x - 3) + 2) >> 2;
            pred[y * n + x] = (uint8_t)v;
        }
        break;
    case 6: if (!(have_left && have_up && have_upleft)) return;   /* Horizontal_Down */
        for (int y = 0; y < n; y++) for (int x = 0; x < n; x++) {
            int z = 2 * y - x, v;
            if (z >= 0 && (z & 1) == 0) v = (L(y - (x >> 1) - 1) + L(y - (x >> 1)) + 1) >> 1;
            else if (z >= 0) v = (L(y - (x >> 1) - 2) + 2 * L(y - (x >> 1) - 1) + L(y - (x >> 1)) + 2) >> 2;
            else if (z == -1) v = (l[0] + 2 * tl + t[0] + 2) >> 2;
            else if (n == 4) v = (T(x - 1) + 2 * T(x - 2) + T(x - 3) + 2) >> 2;
            else v = (T(x - 2 * y - 1) + 2 * T(x - 2 * y - 2) + T(x - 2 * y - 3) + 2) >> 2;
            pred[y * n + x] = (uint8_t)v;
        }
        break;
    case 7: if (!have_up) return;                       /* Vertical_Left */
        for (int y = 0; y < n; y++) for (int x = 0; x < n; x++) {
            int i = x + (y >> 1);
            pred[y * n + x] = (uint8_t)((y & 1) ? (t[i] + 2 * t[i + 1] + t[i + 2] + 2) >> 2 : (t[i] + t[i + 1] + 1) >> 1);
        }
        break;
    case 8: if (!have_left) return;                     /* Horizontal_Up */
        for (int y = 0; y < n; y++) for (int x = 0; x < n; x++) {
            int z = x + 2 * y, i = y + (x >> 1), zmax = 2 * n - 3, v;
            if (z > zmax) v = l[n - 1];
            else if (z == zmax) v = (l[n - 2] + 3 * l[n - 1] + 2) >> 2;
            else if (z & 1) v = (l[i] + 2 * l[i + 1] + l[i + 2] + 2) >> 2;
            else v = (l[i] + l[i + 1] + 1) >> 1;
            pred[y * n + x] = (uint8_t)v;
        }
        break;
    default: break;
    }
#undef T
#undef L
}

/* h264_intra_prediction.c:315-483 */
static void predict_4x4(const uint8_t *pix, int stride, int mode, int have_left, int have_up,
                        int have_upright, uint8_t pred[16])
{
    int t[8] = {0}, l[4] = {0}, tl = 0;
    if (have_left) for (int y = 0; y < 4; y++) l[y] = PX(-1, y);
    if (have_up) {
        for (int x = 0; x < 4; x++) t[x] = PX(x, -1);
        for (int x = 4; x < 8; x++) t[x] = have_upright ? PX(x, -1) : t[3];      /* :431-439 */
    }
    if (have_left && have_up) tl = PX(-1, -1);
    predict_nxn(4, mode, t, l, tl, have_left, have_up, have_left && have_up, pred);
}

/* h264_intra_prediction.c:1107-1283 with the reference sample filter :1295-1353 */
static void predict_8x8(const uint8_t *pix, int stride, int mode, int have_left, int have_up,
                        int have_upleft, int have_upright, uint8_t pred[64])
{
    int t[16] = {0}, l[8] = {0}, tl = 0, ft[16] = {0}, fl[8] = {0}, ftl = 0;
    if (have_left) for (int y = 0; y < 8; y++) l[y] = PX(-1, y);
    if (have_up) {
        for (int x = 0; x < 8; x++) t[x] = PX(x, -1);
        for (int x = 8; x < 16; x++) t[x] = have_upright ? PX(x, -1) : t[7];     /* :1230-1236 */
    }
    if (have_upleft) tl = PX(-1, -1);

    if (have_up) {                                                               /* :1305-1318 */
        ft[0] = have_upleft ? (tl + 2 * t[0] + t[1] + 2) >> 2 : (3 * t[0] + t[1] + 2) >> 2;
        for (int x = 1; x < 15; x++) ft[x] = (t[x - 1] + 2 * t[x] + t[x + 1] + 2) >> 2;
        ft[15] = (t[14] + 3 * t[15] + 2) >> 2;
    }
    if (have_upleft) {                                                           /* :1320-1338 */
        if (have_up && have_left) ftl = (t[0] + 2 * tl + l[0] + 2) >> 2;
        else if (have_up) ftl = (3 * tl + t[0] + 2) >> 2;
        else if (have_left) ftl = (3 * tl + l[0] + 2) >> 2;
        else ftl = tl;
    }
    if (have_left) {                                                             /* :1340-1352 */
        fl[0] = have_upleft ? (tl + 2 * l[0] + l[1] + 2) >> 2 : (3 * l[0] + l[1] + 2) >> 2;
        for (int y = 1; y < 7; y++) fl[y] = (l[y - 1] + 2 * l[y] + l[y + 1] + 2) >> 2;
        fl[7] = (l[6] + 3 * l[7] + 2) >> 2;
    }
    predict_nxn(8, mode, ft, fl, ftl, have_left, have_up, have_upleft, pred);
}

/* h264_intra_prediction.c:1809-2141 */
static void predict_16x16(const uint8_t *pix, int stride, int mode, int have_left, int have_up, uint8_t pred[256])
{
    int t[16] = {0}, l[16] = {0}, tl = 0;
    if (have_up) for (int x = 0; x < 16; x++) t[x] = PX(x, -1);
    if (have_left) for (int y = 0; y < 16; y++) l[y] = PX(-1, y);
    if (have_up && have_left) tl = PX(-1, -1);
    memset(pred, 0, 256);
    if (mode == 0) { if (!have_up) return;
        for (int y = 0; y < 16; y++) for (int x = 0; x < 16; x++) pred[y * 16 + x] = (uint8_t)t[x];
    } else if (mode == 1) { if (!have_left) return;
        for (int y = 0; y < 16; y++) for (int x = 0; x < 16; x++) pred[y * 16 + x] = (uint8_t)l[y];
    } else if (mode == 2) {
        int st = 0, sl = 0, v;
        for (int i = 0; i < 16; i++) { st += t[i]; sl += l[i]; }
        if (have_left && have_up) v = (st + sl + 16) >> 5;
        else if (have_left) v = (sl + 8) >> 4;
        else if (have_up) v = (st + 8) >> 4;
        else v = 128;
        memset(pred, v, 256);
    } else { if (!(have_left && have_up)) return;                               /* Plane :2099-2141 */
        int H = 0, V = 0;
        for (int i = 0; i < 8; i++) {
            H += (i + 1) * (t[8 + i] - (i == 7 ? tl : t[6 - i]));
            V += (i + 1) * (l[8 + i] - (i == 7 ? tl : l[6 - i]));
        }
        int a = 16 * (l[15] + t[15]), b = (5 * H + 32) >> 6, c = (5 * V + 32) >> 6;
        for (int y = 0; y < 16; y++) for (int x = 0; x < 16; x++)
            pred[y * 16 + x] = (uint8_t)clip8((a + b * (x - 7) + c * (y - 7) + 16) >> 5);
    }
}

/* h264_intra_prediction.c:2157-2564, ChromaArrayType 1 */
static void predict_chroma(const uint8_t *pix, int stride, int mode, int have_left, int have_up, uint8_t pred[64])
{
    int t[8] = {0}, l[8] = {0}, tl = 0;
    if (have_up) for (int x = 0; x < 8; x++) t[x] = PX(x, -1);
    if (have_left) for (int y = 0; y < 8; y++) l[y] = PX(-1, y);
    if (have_up && have_left) tl = PX(-1, -1);
    memset(pred, 0, 64);
    if (mode == 0) {                                                             /* DC :2338-2437 */
        for (int blk = 0; blk < 4; blk++) {
            int xo = (blk & 1) * 4, yo = (blk >> 1) * 4, st = 0, sl = 0, v;
            for (int i = 0; i < 4; i++) { st += t[xo + i]; sl += l[yo + i]; }
            if (!have_left && !have_up) v = 128;
            else if ((xo == 0 && yo == 0) || (xo > 0 && yo > 0))
                v = (have_left && have_up) ? (st + sl + 4) >> 3 : have_left ? (sl + 2) >> 2 : (st + 2) >> 2;
            else if (xo > 0) v = have_up ? (st + 2) >> 2 : (sl + 2) >> 2;
            else v = have_left ? (sl + 2) >> 2 : (st + 2) >> 2;
            for (int y = 0; y < 4; y++) for (int x = 0; x < 4; x++) pred[(yo + y) * 8 + xo + x] = (uint8_t)v;
        }
    } else if (mode == 1) { if (!have_left) return;
        for (int y = 0; y < 8; y++) for (int x = 0; x < 8; x++) pred[y * 8 + x] = (uint8_t)l[y];
    } else if (mode == 2) { if (!have_up) return;
        for (int y = 0; y < 8; y++) for (int x = 0; x < 8; x++) pred[y * 8 + x] = (uint8_t)t[x];
    } else { if (!(have_left && have_up)) return;                               /* Plane :2520-2564 */
        int H = 0, V = 0;
        for (int i = 0; i < 4; i++) {
            H += (i + 1) * (t[4 + i] - (i == 3 ? tl : t[2 - i]));
            V += (i + 1) * (l[4 + i] - (i == 3 ? tl : l[2 - i]));
        }
        int a = 16 * (l[7] + t[7]), b = (34 * H + 32) >> 6, c = (34 * V + 32) >> 6;
        for (int y = 0; y < 8; y++) for (int x = 0; x < 8; x++)
            pred[y * 8 + x] = (uint8_t)clip8((a + b * (x - 3) + c * (y - 3) + 16) >> 5);
    }
}
#undef PX

/* kernel 1 hands the residual on as int16 clamped to [-512, 511]: Clip1(pred + r) is the same for any
 * clamp range that contains [-255, 255], and 255 + 511 stays inside a packed 16-bit add */
static inline int16_t sat16(int32_t v) { return (int16_t)(v < -512 ? -512 : (v > 511 ? 511 : v)); }

void oracle_reconstruct_picture(const oracle_sps *sps,
                                const uint8_t *mb_kind, const uint8_t *i16_mode,
                                const uint8_t *chroma_mode, const int8_t *qp_y,
                                const uint8_t *luma_modes, const int16_t *coeff,
                                uint8_t *y, uint8_t *cb, uint8_t *cr, int16_t *residual_out)
{
    int W = sps->width_mbs, H = sps->height_mbs;
    int ys = W * 16, cs = W * 8;
    int32_t res[384];
    uint8_t pred[256];

    for (int my = 0; my < H; my++)
        for (int mx = 0; mx < W; mx++) {
            int a = my * W + mx;
            /* geometric neighbour availability: h264_spatial.c:333-395 */
            int availA = mx > 0, availB = my > 0, availC = my > 0 && mx < W - 1, availD = mx > 0 && my > 0;
            oracle_mb_residual(sps, mb_kind[a], qp_y[a], coeff + (size_t)a * 384, res);
            if (residual_out)
                for (int k = 0; k < 384; k++) residual_out[(size_t)a * 384 + k] = sat16(res[k]);
            uint8_t *py = y + (size_t)(my * 16) * ys + mx * 16;

            if (mb_kind[a] == 0) {                    /* h264_intra_prediction.c:161-177 */
                for (int blk = 0; blk < 16; blk++) {
                    int xo = blk4_x(blk), yo = blk4_y(blk);
                    int left = xo > 0 || availA, up = yo > 0 || availB, upright;
                    /* h264_intra_prediction.c:398-429 + h264_spatial.c:757-774 */
                    if (blk == 3 || blk == 11) upright = 0;
                    else if (yo > 0) upright = xo + 4 < 16;
                    else upright = xo + 4 < 16 ? availB : availC;
                    uint8_t *pb = py + yo * ys + xo;
                    predict_4x4(pb, ys, luma_modes[a * 16 + blk], left, up, upright, pred);
                    for (int i = 0; i < 4; i++)       /* h264_transform.c:150-155, :1419-1421 */
                        for (int j = 0; j < 4; j++)
                            pb[i * ys + j] = (uint8_t)clip8(pred[i * 4 + j] + res[(yo + i) * 16 + xo + j]);
                }
            } else if (mb_kind[a] == 1) {             /* h264_intra_prediction.c:942-958 */
                for (int b8 = 0; b8 < 4; b8++) {
                    int xo = (b8 & 1) * 8, yo = (b8 >> 1) * 8;
                    int left = xo > 0 || availA, up = yo > 0 || availB;
                    int upleft = (xo > 0 && yo > 0) ? 1 : (xo > 0 ? availB : (yo > 0 ? availA : availD));
                    int upright = b8 == 0 ? availB : (b8 == 1 ? availC : (b8 == 2 ? 1 : 0));
                    uint8_t *pb = py + yo * ys + xo;
                    predict_8x8(pb, ys, luma_modes[a * 16 + b8], left, up, upleft, upright, pred);
                    for (int i = 0; i < 8; i++)       /* h264_transform.c:265-270, :1510-1512 */
                        for (int j = 0; j < 8; j++)
                            pb[i * ys + j] = (uint8_t)clip8(pred[i * 8 + j] + res[(yo + i) * 16 + xo + j]);
                }
            } else {                                  /* h264_intra_prediction.c:1809-1932 */
                predict_16x16(py, ys, i16_mode[a], availA, availB, pred);
                for (int i = 0; i < 16; i++)          /* h264_transform.c:216-222 */
                    for (int j = 0; j < 16; j++)
                        py[i * ys + j] = (uint8_t)clip8(pred[i * 16 + j] + res[i * 16 + j]);
            }

            for (int p = 0; p < 2; p++) {             /* h264_intra_prediction.c:2157-2323 */
                uint8_t *pc = (p ? cr : cb) + (size_t)(my * 8) * cs + mx * 8;
                predict_chroma(pc, cs, chroma_mode[a], availA, availB, pred);
                for (int i = 0; i < 8; i++)           /* h264_transform.c:388-400 */
                    for (int j = 0; j < 8; j++)
                        pc[i * cs + j] = (uint8_t)clip8(pred[i * 8 + j] + res[256 + p * 64 + i * 8 + j]);
            }
        }
}

void oracle_yuv420_to_rgb(int width, int height, const uint8_t *y, const uint8_t *cb,
                          const uint8_t *cr, int scale, uint8_t *rgb)
{
    int ow = width / scale, oh = height / scale, area = scale * scale;
    for (int oy = 0; oy < oh; oy++)
        for (int ox = 0; ox < ow; ox++) {
            int acc[3] = {0, 0, 0};
            for (int dy = 0; dy < scale; dy++)
                for (int dx = 0; dx < scale; dx++) {
                    int px = ox * scale + dx, py = oy * scale + dy;
                    int Y = y[py * width + px];
                    int Cb = cb[(py >> 1) * (width >> 1) + (px >> 1)];   /* 2x2 replication, export_utils.c:278-279 */
                    int Cr = cr[(py >> 1) * (width >> 1) + (px >> 1)];
                    int t = (298 * Y) >> 8;                               /* export_utils.c:300-302 */
                    acc[0] += clip8(t + ((408 * Cr) >> 8) - 222);
                    acc[1] += clip8(t - ((100 * Cb) >> 8) - ((208 * Cr) >> 8) + 135);
                    acc[2] += clip8(t + ((516 * Cb) >> 8) - 276);
                }
            uint8_t *o = rgb + ((size_t)oy * ow + ox) * 3;
            for (int k = 0; k < 3; k++) o[k] = (uint8_t)((acc[k] + area / 2) / area);
        }
}
