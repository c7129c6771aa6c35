"""Numpy restatement of the transform stage (spec 8.5), written independently of recon_oracle.c and the kernels.

Every value is an int64 array; wrap() reduces it modulo 2^32 into the int32 range after every operation the decoding
process does in 32 bits (products, left shifts, sums), so the result on hostile levels is defined and the same on every
machine.  residual() returns what mvg_download_residual() and the oracle's residual tap return: per macroblock 256
luma samples (raster, y*16+x), then Cb and Cr (raster, y*8+x), clamped to [-512, 511] as int16.
"""
from __future__ import annotations

import numpy as np


def wrap(x):
    """x modulo 2^32, as a signed 32-bit value (held in int64)."""
    return ((np.asarray(x, np.int64) + 0x80000000) & 0xFFFFFFFF) - 0x80000000


def _scan(n):
    """Zig-zag scan (spec Table 8-13 / 8-14, frame macroblocks): scan index -> raster position, by anti-diagonals,
    odd diagonals walked downwards (row rising), even ones upwards."""
    cells = [(r, c) for r in range(n) for c in range(n)]
    cells.sort(key=lambda rc: (rc[0] + rc[1], rc[0] if (rc[0] + rc[1]) % 2 else rc[1]))
    return np.array([r * n + c for r, c in cells], np.int64)


ZZ4, ZZ8 = _scan(4), _scan(8)

# spec 8.5.9: normAdjust4x4 v[m][0..2] and normAdjust8x8 v[m][0..5]
_V4 = np.array([[10, 16, 13], [11, 18, 14], [13, 20, 16], [14, 23, 18], [16, 25, 20], [18, 29, 23]], np.int64)
_V8 = np.array([[20, 18, 32, 19, 25, 24], [22, 19, 35, 21, 28, 26], [26, 23, 42, 24, 33, 31],
                [28, 25, 45, 26, 35, 33], [32, 28, 51, 30, 40, 38], [36, 32, 58, 34, 46, 43]], np.int64)
# spec Table 8-15: QPC for qPI = 30..51
_QPC = [29, 30, 31, 32, 32, 33, 34, 34, 35, 35, 36, 36, 37, 37, 37, 38, 38, 38, 39, 39, 39, 39]


def _norm4(m, i, j):
    if i % 2 == 0 and j % 2 == 0:
        return _V4[m, 0]
    if i % 2 == 1 and j % 2 == 1:
        return _V4[m, 1]
    return _V4[m, 2]


def _norm8(m, i, j):
    if i % 4 == 0 and j % 4 == 0:
        return _V8[m, 0]
    if i % 2 == 1 and j % 2 == 1:
        return _V8[m, 1]
    if i % 4 == 2 and j % 4 == 2:
        return _V8[m, 2]
    if (i % 4 == 0 and j % 2 == 1) or (i % 2 == 1 and j % 4 == 0):
        return _V8[m, 3]
    if (i % 4 == 0 and j % 4 == 2) or (i % 4 == 2 and j % 4 == 0):
        return _V8[m, 4]
    return _V8[m, 5]


def level_scale(lists4x4, list8x8):
    """(ls4[3,6,16], ls8[6,64]) int32 (spec 8.5.9): weightScale (the zig-zag list put back in raster order) times
    normAdjust.  lists4x4 = intra Y, Cb, Cr 4x4 lists in scan order; None = Flat_4x4 / Flat_8x8 (all 16)."""
    ls4 = np.zeros((3, 6, 16), np.int32)
    ls8 = np.zeros((6, 64), np.int32)
    for c in range(3):
        w = np.full(16, 16, np.int64)
        if lists4x4 is not None:
            w[ZZ4] = np.asarray(lists4x4[c], np.int64)
        for m in range(6):
            ls4[c, m] = [w[i * 4 + j] * _norm4(m, i, j) for i in range(4) for j in range(4)]
    w = np.full(64, 16, np.int64)
    if list8x8 is not None:
        w[ZZ8] = np.asarray(list8x8, np.int64)
    for m in range(6):
        ls8[m] = [w[i * 8 + j] * _norm8(m, i, j) for i in range(8) for j in range(8)]
    return ls4, ls8


def chroma_qp(qp_y, offset):
    """spec 8.5.8 with Table 8-15, 8-bit video: qPI = Clip3(0, 51, QPY + offset)."""
    qpi = np.clip(np.asarray(qp_y, np.int64) + offset, 0, 51)
    return np.where(qpi < 30, qpi, np.array([0] * 30 + _QPC, np.int64)[qpi])


def _dequant4(c, ls, qp, keep_dc):
    """spec 8.5.12.1: c, ls [..., 16] raster; qp broadcasts against c[..., 0]."""
    qp = np.asarray(qp, np.int64)[..., None]
    t = wrap(c * ls)
    up = wrap(t << np.maximum(qp // 6 - 4, 0))
    down = wrap(t + (1 << np.maximum(3 - qp // 6, 0))) >> np.maximum(4 - qp // 6, 0)
    d = np.where(qp >= 24, up, down)
    if keep_dc is not None:
        d[..., 0] = np.where(keep_dc, c[..., 0], d[..., 0])
    return d


def _bfly4(x0, x1, x2, x3):
    """one 1-D pass of spec 8.5.12.2 (equations 8-338..8-345)"""
    e0, e1 = wrap(x0 + x2), wrap(x0 - x2)
    e2, e3 = wrap((x1 >> 1) - x3), wrap(x1 + (x3 >> 1))
    return wrap(e0 + e3), wrap(e1 + e2), wrap(e1 - e2), wrap(e0 - e3)


def _idct4(d):
    """spec 8.5.12.2 on [..., 16] raster blocks -> r [..., 16] (before the clamp)"""
    d = d.reshape(d.shape[:-1] + (4, 4))
    f = np.stack(_bfly4(d[..., 0], d[..., 1], d[..., 2], d[..., 3]), axis=-1)                # rows
    h = np.stack(_bfly4(f[..., 0, :], f[..., 1, :], f[..., 2, :], f[..., 3, :]), axis=-2)    # columns
    return (wrap(h + 32) >> 6).reshape(h.shape[:-2] + (16,))


def _idct8_1d(x):
    """one 1-D pass of spec 8.5.13.2 along the last axis of x [..., 8]"""
    v = [x[..., k] for k in range(8)]
    a0 = wrap(v[0] + v[4])
    a1 = wrap(wrap(wrap(-v[3] + v[5]) - v[7]) - (v[7] >> 1))
    a2 = wrap(v[0] - v[4])
    a3 = wrap(wrap(wrap(v[1] + v[7]) - v[3]) - (v[3] >> 1))
    a4 = wrap((v[2] >> 1) - v[6])
    a5 = wrap(wrap(wrap(-v[1] + v[7]) + v[5]) + (v[5] >> 1))
    a6 = wrap(v[2] + (v[6] >> 1))
    a7 = wrap(wrap(wrap(v[3] + v[5]) + v[1]) + (v[1] >> 1))
    b0, b1, b2, b3 = wrap(a0 + a6), wrap(a1 + (a7 >> 2)), wrap(a2 + a4), wrap(a3 + (a5 >> 2))
    b4, b5, b6, b7 = wrap(a2 - a4), wrap((a3 >> 2) - a5), wrap(a0 - a6), wrap(a7 - (a1 >> 2))
    return np.stack([wrap(b0 + b7), wrap(b2 + b5), wrap(b4 + b3), wrap(b6 + b1),
                     wrap(b6 - b1), wrap(b4 - b3), wrap(b2 - b5), wrap(b0 - b7)], axis=-1)


def _hadamard4(m):
    """H m H with H = [[1,1,1,1],[1,1,-1,-1],[1,-1,-1,1],[1,-1,1,-1]] (spec 8-320), m [..., 4, 4]"""
    def pass_(a, b, c, d):
        return wrap(a + b + c + d), wrap(a + b - c - d), wrap(a - b - c + d), wrap(a - b + c - d)
    t = np.stack(pass_(m[..., 0, :], m[..., 1, :], m[..., 2, :], m[..., 3, :]), axis=-2)    # H m
    return np.stack(pass_(t[..., 0], t[..., 1], t[..., 2], t[..., 3]), axis=-1)             # (H m) H


def _blk4_xy(blk):
    """upper-left luma sample of 4x4 block luma4x4BlkIdx (spec 6.4.3)"""
    return 8 * ((blk // 4) % 2) + 4 * ((blk % 4) % 2), 8 * ((blk // 4) // 2) + 4 * ((blk % 4) // 2)


def residual(soa, ls4, ls8):
    """The residual of every macroblock of `soa` (mvgpu.h SoA: coeff [M, 384] in scan order, 24 blocks of 16 then
    four 8x8 blocks of 64 for Intra8x8) with the LevelScale tables (ls4[3,6,16], ls8[6,64]).  [M, 384] int16."""
    coeff = np.asarray(soa.coeff, np.int64)
    kind = np.asarray(soa.mb_kind, np.int64)
    qp = np.asarray(soa.qp_y, np.int64)
    ls4 = np.asarray(ls4, np.int64).reshape(3, 6, 16)
    ls8 = np.asarray(ls8, np.int64).reshape(6, 64)
    M = coeff.shape[0]
    out = np.zeros((M, 384), np.int64)
    luma = out[:, :256].reshape(M, 16, 16)

    # Intra16x16 luma DC (spec 8.5.10): c[i][j] = the level in slot 0 of the block at (4j, 4i)
    lsY = ls4[0][qp % 6]                                                     # [M, 16]
    dcm = np.zeros((M, 4, 4), np.int64)
    for blk in range(16):
        x, y = _blk4_xy(blk)
        dcm[:, y // 4, x // 4] = coeff[:, blk * 16]
    f = _hadamard4(dcm)
    q6 = (qp // 6)[:, None, None]
    t = wrap(f * lsY[:, 0, None, None])
    dcY = np.where(q6 >= 6, wrap(t << np.maximum(q6 - 6, 0)),
                   wrap(t + (1 << np.maximum(5 - q6, 0))) >> np.maximum(6 - q6, 0))

    # 4x4 luma blocks (Intra4x4 and Intra16x16)
    is16 = kind == 2
    for blk in range(16):
        c = np.zeros((M, 16), np.int64)
        c[:, ZZ4] = coeff[:, blk * 16:blk * 16 + 16]
        x, y = _blk4_xy(blk)
        c[:, 0] = np.where(is16, dcY[:, y // 4, x // 4], c[:, 0])
        r = _idct4(_dequant4(c, lsY, qp, is16)).reshape(M, 4, 4)
        sel = kind != 1
        luma[sel, y:y + 4, x:x + 4] = r[sel]

    # 8x8 luma blocks (Intra8x8, spec 8.5.13)
    sel = kind == 1
    if sel.any():
        q8, c8 = qp[sel], coeff[sel]
        for b8 in range(4):
            c = np.zeros((len(q8), 64), np.int64)
            c[:, ZZ8] = c8[:, b8 * 64:b8 * 64 + 64]
            t = wrap(c * ls8[q8 % 6])
            s = (q8 // 6)[:, None]
            d = np.where(s >= 6, wrap(t << np.maximum(s - 6, 0)),
                         wrap(t + (1 << np.maximum(5 - s, 0))) >> np.maximum(6 - s, 0)).reshape(-1, 8, 8)
            g = _idct8_1d(d)                                                    # rows
            h = np.swapaxes(_idct8_1d(np.swapaxes(g, -1, -2)), -1, -2)          # columns
            x, y = 8 * (b8 % 2), 8 * (b8 // 2)
            luma[sel, y:y + 8, x:x + 8] = wrap(h + 32) >> 6

    # chroma (spec 8.5.11): 2x2 DC transform, then the 4x4 blocks with the DC kept
    for p, off in enumerate((soa.cb_qp_offset, soa.cr_qp_offset)):
        qpc = chroma_qp(qp, off)
        ls = ls4[p + 1][qpc % 6]
        cc = coeff[:, 256 + 64 * p:320 + 64 * p]
        c00, c01, c10, c11 = cc[:, 0], cc[:, 16], cc[:, 32], cc[:, 48]
        f = [wrap(c00 + c01 + c10 + c11), wrap(c00 - c01 + c10 - c11),
             wrap(c00 + c01 - c10 - c11), wrap(c00 - c01 - c10 + c11)]          # [[1,1],[1,-1]] c [[1,1],[1,-1]]
        plane = out[:, 256 + 64 * p:320 + 64 * p].reshape(M, 8, 8)
        for blk in range(4):
            dc = wrap(wrap(f[blk] * ls[:, 0]) << (qpc // 6)) >> 5
            c = np.zeros((M, 16), np.int64)
            c[:, ZZ4] = cc[:, blk * 16:blk * 16 + 16]
            c[:, 0] = dc
            r = _idct4(_dequant4(c, ls, qpc, np.ones(M, bool))).reshape(M, 4, 4)
            x, y = 4 * (blk % 2), 4 * (blk // 2)
            plane[:, y:y + 4, x:x + 4] = r
    return np.clip(out, -512, 511).astype(np.int16)
