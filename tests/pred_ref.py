"""Restatement of intra prediction and reconstruction (spec 8.3.1.2, 8.3.2.2, 8.3.3, 8.3.4 for ChromaArrayType 1),
written from the spec independently of recon_oracle.c and the kernels.

Neighbour availability is geometric, as the project decodes it: one slice per picture, every macroblock intra,
constrained_intra_pred_flag = 0.  A sample is available when the macroblock that holds it exists (spec 6.4.12) and,
inside the current macroblock, when its block precedes the current block in decoding order.  The second rule is what the
spec spells out as "x > 3 and luma4x4BlkIdx is 3 or 11" for Intra4x4; for Intra8x8 it leaves the up-right samples of
block 2 (the bottom row of block 1) available and those of block 3 missing.

reconstruct() returns the packed YUV of cpu.reconstruct(): per picture the luma plane, then Cb, then Cr, each in raster
order.  No case was found where the spec and the reference decoder disagree on a conforming stream.

MUTATIONS names plausible implementation mistakes that reconstruct(..., mutation=name) emulates, so that tests can show
which inputs would catch them.
"""
from __future__ import annotations

import numpy as np

import xform_ref

MUTATIONS = (
    "i4_blk5_upright_from_B",       # Intra4x4 block 5 takes its up-right availability from B instead of C
    "i4_blk7_has_upright",          # Intra4x4 block 7 reads p[4..7,-1] as if they were available
    "i8_blk2_no_upright",           # Intra8x8 block 2 substitutes p[7,-1] for its up-right samples
    "i8_p15_unfiltered",            # the 8.3.2.2.1 filter leaves p'[15,-1] = p[15,-1]
    "chroma_dc_rules_swapped",      # chroma DC of the blocks at (4,0) and (0,4) use each other's rule
    "i16_dc_one_side_rounding",     # Intra16x16 DC with one side missing rounds with 16 as with both sides
    "chroma_plane_luma_constant",   # chroma plane uses 5 (luma) instead of 34 in b and c
)


def _blk4_xy(blk):
    """upper-left sample of luma4x4BlkIdx inside the macroblock (spec 6.4.3)"""
    return xform_ref._blk4_xy(blk)


def _blk4_at(x, y):
    """luma4x4BlkIdx of the block that holds sample (x, y) of the macroblock (spec 6.4.13.1)"""
    return 8 * (y // 8) + 4 * (x // 8) + 2 * ((y % 8) // 4) + (x % 8) // 4


class _Picture:
    """The planes being reconstructed and the geometric availability of one picture."""

    def __init__(self, w_mbs, h_mbs):
        self.W, self.H = w_mbs, h_mbs
        self.y = np.zeros((16 * h_mbs, 16 * w_mbs), np.int64)
        self.c = [np.zeros((8 * h_mbs, 8 * w_mbs), np.int64) for _ in range(2)]

    def sample(self, x, y):
        """luma sample (x, y); 0 outside the picture, where only a mutation reads"""
        return int(self.y[y, x]) if 0 <= x < self.y.shape[1] and 0 <= y < self.y.shape[0] else 0

    def mb_available(self, mx, my, xn, yn, size):
        """spec 6.4.12 for a location (xn, yn) relative to macroblock (mx, my) of `size` x `size` samples: is the
        macroblock that holds it available (A, B, C, D by picture geometry); inside the current one -> None."""
        if 0 <= xn < size and 0 <= yn < size:
            return None
        if xn < 0 and yn < 0:
            return mx > 0 and my > 0                        # D
        if xn < 0 and 0 <= yn < size:
            return mx > 0                                   # A
        if 0 <= xn < size and yn < 0:
            return my > 0                                   # B
        if xn >= size and yn < 0:
            return my > 0 and mx < self.W - 1               # C
        return False                                        # right of or below the current macroblock


def _nxn_neighbours(pic, mx, my, n, blk, xo, yo, mutation):
    """p[x, -1] (x = -1..2n-1) and p[-1, y] (y = 0..n-1) of an n x n luma block at (xo, yo) of macroblock (mx, my),
    None where not available, after the substitution of p[n-1, -1] for missing up-right samples."""
    X, Y = 16 * mx + xo, 16 * my + yo

    def avail(xn, yn):
        a = pic.mb_available(mx, my, xn, yn, 16)
        if a is not None:
            return a
        return (_blk4_at(xn, yn) if n == 4 else 2 * (yn // 8) + xn // 8) < blk      # decoded before this block

    top = {}
    for x in range(-1, 2 * n):
        ok = avail(xo + x, yo - 1)
        if x >= n:
            if mutation == "i4_blk5_upright_from_B" and n == 4 and blk == 5:
                ok = my > 0
            elif mutation == "i4_blk7_has_upright" and n == 4 and blk == 7:
                ok = True
            elif mutation == "i8_blk2_no_upright" and n == 8 and blk == 2:
                ok = False
        top[x] = pic.sample(X + x, Y - 1) if ok else None
    if top[n - 1] is not None:
        for x in range(n, 2 * n):
            if top[x] is None:
                top[x] = top[n - 1]
    left = {y: (pic.sample(X - 1, Y + y) if avail(xo - 1, yo + y) else None) for y in range(n)}
    return top, left


def _filter8(top, left, mutation):
    """spec 8.3.2.2.1: reference sample filtering of the Intra8x8 neighbour line."""
    t, l, tl = top, left, top[-1]
    ft, fl, ftl = {x: None for x in range(16)}, {y: None for y in range(8)}, None
    if all(t[x] is not None for x in range(16)):
        ft[0] = (tl + 2 * t[0] + t[1] + 2) >> 2 if tl is not None else (3 * t[0] + t[1] + 2) >> 2
        for x in range(1, 15):
            ft[x] = (t[x - 1] + 2 * t[x] + t[x + 1] + 2) >> 2
        ft[15] = t[15] if mutation == "i8_p15_unfiltered" else (t[14] + 3 * t[15] + 2) >> 2
    if tl is not None:
        # with geometric availability in one slice, D present implies A and B present: the three partial branches
        # below are the spec's and cannot be reached by a conforming picture of this project
        if t[0] is None or l[0] is None:
            if t[0] is not None:
                ftl = (3 * tl + t[0] + 2) >> 2
            elif l[0] is not None:
                ftl = (3 * tl + l[0] + 2) >> 2
            else:
                ftl = tl
        else:
            ftl = (t[0] + 2 * tl + l[0] + 2) >> 2
    if all(l[y] is not None for y in range(8)):
        fl[0] = (tl + 2 * l[0] + l[1] + 2) >> 2 if tl is not None else (3 * l[0] + l[1] + 2) >> 2
        for y in range(1, 7):
            fl[y] = (l[y - 1] + 2 * l[y] + l[y + 1] + 2) >> 2
        fl[7] = (l[6] + 3 * l[7] + 2) >> 2
    ft[-1] = ftl
    return ft, fl


def _predict_nxn(n, mode, top, left):
    """spec 8.3.1.2.1..9 (n = 4) and 8.3.2.2.2..10 (n = 8, on the filtered samples): pred[y][x]."""
    def P(x, y):
        v = top[x] if y == -1 else left[y] if x == -1 else None
        assert v is not None, (n, mode, x, y)           # a mode that reads a missing sample is not conforming
        return v

    has_top = all(top[x] is not None for x in range(n))
    has_left = all(left[y] is not None for y in range(n))
    zmax = 2 * n - 3                                     # zHU of the one sample that blends p[-1, n-2] and p[-1, n-1]
    k = 2 if n == 4 else 3                               # log2(n)
    out = [[0] * n for _ in range(n)]
    for y in range(n):
        for x in range(n):
            if mode == 0:
                v = P(x, -1)
            elif mode == 1:
                v = P(-1, y)
            elif mode == 2:
                st = sum(top[i] for i in range(n)) if has_top else 0
                sl = sum(left[i] for i in range(n)) if has_left else 0
                if has_top and has_left:
                    v = (st + sl + n) >> (k + 1)
                elif has_left:
                    v = (sl + (n >> 1)) >> k
                elif has_top:
                    v = (st + (n >> 1)) >> k
                else:
                    v = 128
            elif mode == 3:
                if x == n - 1 and y == n - 1:
                    v = (P(2 * n - 2, -1) + 3 * P(2 * n - 1, -1) + 2) >> 2
                else:
                    v = (P(x + y, -1) + 2 * P(x + y + 1, -1) + P(x + y + 2, -1) + 2) >> 2
            elif mode == 4:
                if x > y:
                    v = (P(x - y - 2, -1) + 2 * P(x - y - 1, -1) + P(x - y, -1) + 2) >> 2
                elif x < y:
                    v = (P(-1, y - x - 2) + 2 * P(-1, y - x - 1) + P(-1, y - x) + 2) >> 2
                else:
                    v = (P(0, -1) + 2 * P(-1, -1) + P(-1, 0) + 2) >> 2
            elif mode == 5:
                z = 2 * x - y
                if z >= 0 and z % 2 == 0:
                    v = (P(x - (y >> 1) - 1, -1) + P(x - (y >> 1), -1) + 1) >> 1
                elif z >= 0:
                    v = (P(x - (y >> 1) - 2, -1) + 2 * P(x - (y >> 1) - 1, -1) + P(x - (y >> 1), -1) + 2) >> 2
                elif z == -1:
                    v = (P(-1, 0) + 2 * P(-1, -1) + P(0, -1) + 2) >> 2
                else:
                    v = (P(-1, y - 2 * x - 1) + 2 * P(-1, y - 2 * x - 2) + P(-1, y - 2 * x - 3) + 2) >> 2
            elif mode == 6:
                z = 2 * y - x
                if z >= 0 and z % 2 == 0:
                    v = (P(-1, y - (x >> 1) - 1) + P(-1, y - (x >> 1)) + 1) >> 1
                elif z >= 0:
                    v = (P(-1, y - (x >> 1) - 2) + 2 * P(-1, y - (x >> 1) - 1) + P(-1, y - (x >> 1)) + 2) >> 2
                elif z == -1:
                    v = (P(-1, 0) + 2 * P(-1, -1) + P(0, -1) + 2) >> 2
                else:
                    v = (P(x - 2 * y - 1, -1) + 2 * P(x - 2 * y - 2, -1) + P(x - 2 * y - 3, -1) + 2) >> 2
            elif mode == 7:
                i = x + (y >> 1)
                if y % 2 == 0:
                    v = (P(i, -1) + P(i + 1, -1) + 1) >> 1
                else:
                    v = (P(i, -1) + 2 * P(i + 1, -1) + P(i + 2, -1) + 2) >> 2
            elif mode == 8:
                z, i = x + 2 * y, y + (x >> 1)
                if z > zmax:
                    v = P(-1, n - 1)
                elif z == zmax:
                    v = (P(-1, n - 2) + 3 * P(-1, n - 1) + 2) >> 2
                elif z % 2 == 0:
                    v = (P(-1, i) + P(-1, i + 1) + 1) >> 1
                else:
                    v = (P(-1, i) + 2 * P(-1, i + 1) + P(-1, i + 2) + 2) >> 2
            else:
                raise ValueError(f"Intra{n}x{n} mode {mode}")
            out[y][x] = v
    return np.array(out, np.int64)


def _plane(a, b, c, size, centre):
    """Clip1((a + b * (x - centre) + c * (y - centre) + 16) >> 5) over a size x size block"""
    xs = np.arange(size, dtype=np.int64)
    return np.clip((a + b * (xs[None, :] - centre) + c * (xs[:, None] - centre) + 16) >> 5, 0, 255)


def _predict_16x16(pic, mx, my, mode, mutation):
    """spec 8.3.3"""
    X, Y = 16 * mx, 16 * my
    has_top, has_left = my > 0, mx > 0
    t = pic.y[Y - 1, X:X + 16] if has_top else None
    l = pic.y[Y:Y + 16, X - 1] if has_left else None
    if mode == 0:
        return np.repeat(t[None, :], 16, 0)
    if mode == 1:
        return np.repeat(l[:, None], 16, 1)
    if mode == 2:
        one = 16 if mutation == "i16_dc_one_side_rounding" else 8
        if has_top and has_left:
            v = (int(t.sum()) + int(l.sum()) + 16) >> 5
        elif has_left:
            v = (int(l.sum()) + one) >> 4
        elif has_top:
            v = (int(t.sum()) + one) >> 4
        else:
            v = 128
        return np.full((16, 16), v, np.int64)
    if mode == 3:
        tl = int(pic.y[Y - 1, X - 1])
        p_top = lambda x: tl if x < 0 else int(t[x])
        p_left = lambda y: tl if y < 0 else int(l[y])
        H = sum((i + 1) * (p_top(8 + i) - p_top(6 - i)) for i in range(8))
        V = sum((i + 1) * (p_left(8 + i) - p_left(6 - i)) for i in range(8))
        a = 16 * (int(l[15]) + int(t[15]))
        return _plane(a, (5 * H + 32) >> 6, (5 * V + 32) >> 6, 16, 7)
    raise ValueError(f"Intra16x16 mode {mode}")


def _predict_chroma(pic, plane, mx, my, mode, mutation):
    """spec 8.3.4 with ChromaArrayType 1 (MbWidthC = MbHeightC = 8, xCF = yCF = 0)"""
    X, Y = 8 * mx, 8 * my
    src = pic.c[plane]
    has_top, has_left = my > 0, mx > 0
    t = src[Y - 1, X:X + 8] if has_top else None
    l = src[Y:Y + 8, X - 1] if has_left else None
    if mode == 0:
        out = np.zeros((8, 8), np.int64)
        for blk in range(4):
            xo, yo = 4 * (blk % 2), 4 * (blk // 2)
            st = int(t[xo:xo + 4].sum()) if has_top else None
            sl = int(l[yo:yo + 4].sum()) if has_left else None
            rule = "corner" if (xo, yo) in ((0, 0), (4, 4)) else "top" if yo == 0 else "left"
            if mutation == "chroma_dc_rules_swapped" and rule != "corner":
                rule = "left" if rule == "top" else "top"
            if rule == "corner":
                v = ((st + sl + 4) >> 3 if st is not None and sl is not None else
                     (sl + 2) >> 2 if sl is not None else (st + 2) >> 2 if st is not None else 128)
            elif rule == "top":
                v = (st + 2) >> 2 if st is not None else (sl + 2) >> 2 if sl is not None else 128
            else:
                v = (sl + 2) >> 2 if sl is not None else (st + 2) >> 2 if st is not None else 128
            out[yo:yo + 4, xo:xo + 4] = v
        return out
    if mode == 1:
        return np.repeat(l[:, None], 8, 1)
    if mode == 2:
        return np.repeat(t[None, :], 8, 0)
    if mode == 3:
        tl = int(src[Y - 1, X - 1])
        p_top = lambda x: tl if x < 0 else int(t[x])
        p_left = lambda y: tl if y < 0 else int(l[y])
        H = sum((i + 1) * (p_top(4 + i) - p_top(2 - i)) for i in range(4))
        V = sum((i + 1) * (p_left(4 + i) - p_left(2 - i)) for i in range(4))
        k = 5 if mutation == "chroma_plane_luma_constant" else 34
        a = 16 * (int(l[7]) + int(t[7]))
        return _plane(a, (k * H + 32) >> 6, (k * V + 32) >> 6, 8, 3)
    raise ValueError(f"chroma mode {mode}")


def _reconstruct_mb(pic, soa, a, mx, my, res, mutation):
    kind = int(soa.mb_kind[a])
    X, Y = 16 * mx, 16 * my
    r = res[a].astype(np.int64)
    luma_res = r[:256].reshape(16, 16)
    if kind == 0:
        for blk in range(16):
            xo, yo = _blk4_xy(blk)
            top, left = _nxn_neighbours(pic, mx, my, 4, blk, xo, yo, mutation)
            pred = _predict_nxn(4, int(soa.luma_modes[a, blk]), top, left)
            pic.y[Y + yo:Y + yo + 4, X + xo:X + xo + 4] = np.clip(pred + luma_res[yo:yo + 4, xo:xo + 4], 0, 255)
    elif kind == 1:
        for b8 in range(4):
            xo, yo = 8 * (b8 % 2), 8 * (b8 // 2)
            top, left = _filter8(*_nxn_neighbours(pic, mx, my, 8, b8, xo, yo, mutation), mutation)
            pred = _predict_nxn(8, int(soa.luma_modes[a, b8]), top, left)
            pic.y[Y + yo:Y + yo + 8, X + xo:X + xo + 8] = np.clip(pred + luma_res[yo:yo + 8, xo:xo + 8], 0, 255)
    elif kind == 2:
        pred = _predict_16x16(pic, mx, my, int(soa.i16_mode[a]), mutation)
        pic.y[Y:Y + 16, X:X + 16] = np.clip(pred + luma_res, 0, 255)
    else:
        raise ValueError(f"macroblock kind {kind}")
    for p in range(2):
        pred = _predict_chroma(pic, p, mx, my, int(soa.chroma_mode[a]), mutation)
        c_res = r[256 + 64 * p:320 + 64 * p].reshape(8, 8)
        pic.c[p][8 * my:8 * my + 8, 8 * mx:8 * mx + 8] = np.clip(pred + c_res, 0, 255)


def reconstruct(soa, ls4, ls8, mutation=None):
    """The decoded pictures of `soa` with the LevelScale tables (ls4[3,6,16], ls8[6,64]): [P, 1.5 * W * H] uint8, the
    layout of cpu.reconstruct().  `mutation` (one of MUTATIONS) emulates a mistake."""
    assert mutation is None or mutation in MUTATIONS, mutation
    res = xform_ref.residual(soa, ls4, ls8)
    W, H, N = soa.width_mbs, soa.height_mbs, soa.n_mbs
    out = np.zeros((soa.n_pics, 256 * N * 3 // 2), np.uint8)
    for p in range(soa.n_pics):
        pic = _Picture(W, H)
        for my in range(H):
            for mx in range(W):
                _reconstruct_mb(pic, soa, p * N + my * W + mx, mx, my, res, mutation)
        out[p] = np.concatenate([pic.y.ravel(), pic.c[0].ravel(), pic.c[1].ravel()])
    return out
