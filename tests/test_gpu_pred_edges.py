"""Intra prediction in every (kind, block, mode, availA, availB, availC) case a conforming picture can contain, on
hand-built SoAs, checked against the oracle and against pred_ref.py (a restatement of spec 8.3).

Layout.  Test macroblocks sit on even rows, on every other column (shifted by one from one test row to the next), so
that their A, B, C and D neighbours are texture macroblocks: random legal modes and random levels.  Intra16x16 test
macroblocks have all levels zero, so that their output is the prediction itself.  Intra4x4 and Intra8x8 test
macroblocks carry zero levels in their test blocks only: every other block in both directions (4 of the 16 4x4 blocks,
1 of the 4 8x8 blocks), the rest carrying random levels.  A block that reads only samples of its own macroblock would
otherwise read flat predictions (128 everywhere in the first macroblock of a picture), where a wrong tap cannot show;
this way every neighbour a test block reads is textured.  Chroma levels of test macroblocks are zero.

Cases:
- `coverage_*`: every legal combination, at least REPEATS times as a test block, in pictures 1, 2, 3, 6 and 13
  macroblocks wide (one-wide pictures are the only ones with B present and A and C missing; widths 6 and 13 end in a
  short group of the fused kernel's four-macroblock halo groups).
- `upright_halo`: Intra4x4 block 5 and Intra8x8 block 1 in modes 3 and 7, whose up-right samples lie in macroblock C,
  at every column position modulo 4 and in the short last group, with and without C.
- `mixed_i4`: Intra4x4 mode words drawn at random among the legal modes, so that the two blocks of a diagonal step mix
  DC (both sides, and picture-edge DC) with directional modes.
- `sat_*` (allowed to clip, kept apart): Intra16x16 and chroma plane next to 0...0 / 255...255 steps, where |b| and |c|
  reach 717 and 1355 and the plane clips below 0 and above 255 inside one macroblock; every mode on all-0 and all-255
  neighbours.
"""
from collections import Counter

import numpy as np
import pytest

import pred_ref
from minivideo_b200.synth import Soa

I4, I8, I16 = 0, 1, 2
QP = 28
REPEATS = 3
TRIPLES = ((0, 0, 0), (1, 0, 0), (0, 1, 1), (0, 1, 0), (1, 1, 1), (1, 1, 0))     # (availA, availB, availC)
LEGAL_COMBINATIONS = 942


# ---------------------------------------------------------------------------------------------------------------------
# legality (spec 7.4.5 / the modes pick_nxn_mode and pick_16_mode of h264_synth.c draw)

def _nxn_legal(left, up):
    return [m for m in range(9) if not ((m in (0, 3, 7) and not up) or (m in (1, 8) and not left)
                                        or (4 <= m <= 6 and not (left and up)))]


def _i16_legal(left, up):
    """Intra16x16 0 V, 1 H, 2 DC, 3 Plane"""
    return [m for m in range(4) if not ((m == 0 and not up) or (m == 1 and not left) or (m == 3 and not (left and up)))]


def _chroma_legal(left, up):
    """chroma 0 DC, 1 H, 2 V, 3 Plane"""
    return [m for m in range(4) if not ((m == 2 and not up) or (m == 1 and not left) or (m == 3 and not (left and up)))]


def _origin(n, blk):
    return pred_ref._blk4_xy(blk) if n == 4 else (8 * (blk % 2), 8 * (blk // 2))


def _block_legal(n, blk, a, b):
    xo, yo = _origin(n, blk)
    return _nxn_legal(xo > 0 or a, yo > 0 or b)


def _upright(n, blk, a, b, c):
    """are the up-right samples p[n..2n-1, -1] of the block available (spec 6.4.12, decoding order inside the MB)"""
    xo, yo = _origin(n, blk)
    xr, yr = xo + n, yo - 1
    if yr < 0:
        return bool(b if xr < 16 else c)
    if xr >= 16:
        return False
    return (pred_ref._blk4_at(xr, yr) if n == 4 else 2 * (yr // 8) + xr // 8) < blk


def combination(kind, blk, mode, a, b, c):
    """The key of a case: Intra16x16 and chroma prediction never read macroblock C, so availC is not part of theirs."""
    return (kind, blk, mode, a, b, c if kind in ("i4", "i8") else None)


def legal_combinations():
    out = set()
    for a, b, c in TRIPLES:
        for blk in range(16):
            out |= {combination("i4", blk, m, a, b, c) for m in _block_legal(4, blk, a, b)}
        for b8 in range(4):
            out |= {combination("i8", b8, m, a, b, c) for m in _block_legal(8, b8, a, b)}
        out |= {combination("i16", 0, m, a, b, c) for m in _i16_legal(a, b)}
        out |= {combination("chroma", 0, m, a, b, c) for m in _chroma_legal(a, b)}
    return out


# ---------------------------------------------------------------------------------------------------------------------
# macroblocks

def _levels(rng, n, amp=2, density=0.4):
    return (rng.integers(-amp, amp + 1, n) * (rng.random(n) < density)).astype(np.int16)


def _mb(kind, modes=None, i16=2, chroma=0, coeff=None):
    m = np.zeros(16, np.uint8)
    if modes is not None:
        m[:len(modes)] = modes
    return dict(kind=kind, modes=m, i16=i16, chroma=chroma,
                coeff=np.zeros(384, np.int16) if coeff is None else coeff, tests=[])


def _texture_mb(rng, a, b):
    """random kind, random legal modes, random levels everywhere"""
    kind = int(rng.choice([I4, I8, I16], p=[0.5, 0.3, 0.2]))
    if kind == I16:
        modes = None
    else:
        n = 4 if kind == I4 else 8
        modes = [int(rng.choice(_block_legal(n, k, a, b))) for k in range(16 if n == 4 else 4)]
    return _mb(kind, modes, int(rng.choice(_i16_legal(a, b))), int(rng.choice(_chroma_legal(a, b))),
               _levels(rng, 384))


def _test_blocks(n, off):
    """the blocks of an n x n kind that carry no levels: one in two in each direction, starting at off = (ox, oy)"""
    return [blk for blk in range(16 if n == 4 else 4)
            if (_origin(n, blk)[0] // n) % 2 == off[0] and (_origin(n, blk)[1] // n) % 2 == off[1]]


def _nxn_test_mb(rng, n, modes, off, chroma):
    kind = I4 if n == 4 else I8
    coeff = np.zeros(384, np.int16)
    tests = _test_blocks(n, off)
    size = 16 if n == 4 else 64
    for blk in range(16 if n == 4 else 4):
        if blk not in tests:
            coeff[blk * size:(blk + 1) * size] = _levels(rng, size)
    mb = _mb(kind, modes, chroma=chroma, coeff=coeff)
    mb["tests"] = [("i4" if n == 4 else "i8", blk, int(modes[blk])) for blk in tests] + [("chroma", 0, chroma)]
    return mb


def _i16_test_mb(mode, chroma):
    mb = _mb(I16, None, mode, chroma)
    mb["tests"] = [("i16", 0, mode), ("chroma", 0, chroma)]
    return mb


OFFSETS = ((0, 0), (1, 0), (0, 1), (1, 1))


def _coverage_schedule(triple):
    """One round of test-macroblock recipes for a neighbour availability: together they put every legal mode in every
    block as a test block once."""
    a, b, _ = triple
    out = []
    for n in (4, 8):
        nblk = 16 if n == 4 else 4
        legal = [_block_legal(n, blk, a, b) for blk in range(nblk)]
        for off in OFFSETS:
            tests = _test_blocks(n, off)
            for k in range(max(len(legal[blk]) for blk in tests)):
                out.append(("nxn", n, [legal[blk][(k + blk) % len(legal[blk])] for blk in range(nblk)], off))
    out += [("i16", m) for m in _i16_legal(a, b)]
    return out


def _is_test_position(mx, my):
    return my % 2 == 0 and mx % 2 == (my // 2) % 2


def _batch(w, h, n_pics, content, seed):
    """n_pics pictures of w x h macroblocks; content(rng, pic, mx, my, a, b, c) returns the test macroblock at test
    positions (None: texture).  Returns (Soa, [(pic, mx, my, (a, b, c), kind, block, mode)] of the test blocks)."""
    rng = np.random.default_rng(seed)
    mbs, tests = [], []
    for p in range(n_pics):
        for my in range(h):
            for mx in range(w):
                a, b, c = int(mx > 0), int(my > 0), int(my > 0 and mx < w - 1)
                mb = content(rng, p, mx, my, a, b, c) if _is_test_position(mx, my) else None
                if mb is None:
                    mb = _texture_mb(rng, a, b)
                tests += [(p, mx, my, (a, b, c)) + t for t in mb["tests"]]
                mbs.append(mb)
    n = len(mbs)
    soa = Soa(w, h, n_pics, np.array([m["kind"] for m in mbs], np.uint8), np.array([m["i16"] for m in mbs], np.uint8),
              np.array([m["chroma"] for m in mbs], np.uint8), np.full(n, QP, np.int8), np.full(n, 0x2F, np.uint8),
              np.stack([m["modes"] for m in mbs]), np.stack([m["coeff"] for m in mbs]))
    return soa, tests


# geometry (w, h, pictures) of each coverage batch: the first macroblock of a picture is the only position with
# neither A nor B, the top row the only one with A alone, one-wide pictures the only ones with B alone
COVERAGE_GEOMETRIES = {
    "coverage_w1": (1, 9, 120),
    "coverage_w2": (2, 9, 64),
    "coverage_w3": (3, 9, 40),
    "coverage_w6": (6, 5, 12),
    "coverage_w13": (13, 5, 12),
    "coverage_w13_top_row": (13, 1, 40),
}


def _coverage_cases():
    """All coverage batches, built together: each availability has its own round-robin over its schedule and over the
    legal chroma modes, carried from one batch to the next."""
    state = {t: [0, 0] for t in TRIPLES}

    def content(rng, p, mx, my, a, b, c):
        st = state[(a, b, c)]
        sched = _coverage_schedule((a, b, c))
        chroma_modes = _chroma_legal(a, b)
        recipe, chroma = sched[st[0] % len(sched)], chroma_modes[st[1] % len(chroma_modes)]
        st[0] += 1
        st[1] += 1
        if recipe[0] == "i16":
            return _i16_test_mb(recipe[1], chroma)
        return _nxn_test_mb(rng, recipe[1], recipe[2], recipe[3], chroma)

    return {name: _batch(w, h, n, content, seed=1000 + i)
            for i, (name, (w, h, n)) in enumerate(COVERAGE_GEOMETRIES.items())}


def _halo_case():
    """Intra4x4 block 5 and Intra8x8 block 1 in modes 3 and 7 at every test position of pictures 6 and 13 wide."""
    recipes = [(n, m) for n in (4, 8) for m in (3, 7)]
    count = [0]

    def content(rng, p, mx, my, a, b, c):
        if not b:
            return None
        n, mode = recipes[(count[0] + mx // 2) % 4]
        count[0] += 1
        blk = 5 if n == 4 else 1
        modes = [int(rng.choice(_block_legal(n, k, a, b))) for k in range(16 if n == 4 else 4)]
        modes[blk] = mode
        return _nxn_test_mb(rng, n, modes, (1, 0), int(rng.choice(_chroma_legal(a, b))))

    s6, t6 = _batch(6, 7, 6, content, seed=2001)
    s13, t13 = _batch(13, 7, 6, content, seed=2002)
    return {"upright_halo_w6": (s6, t6), "upright_halo_w13": (s13, t13)}


def _mixed_case():
    """Intra4x4 test macroblocks whose 16 modes are a seeded draw of legal modes, DC drawn with weight 1/3."""
    def content(rng, p, mx, my, a, b, c):
        modes = []
        for blk in range(16):
            legal = _block_legal(4, blk, a, b)
            modes.append(2 if rng.random() < 1 / 3 else int(rng.choice(legal)))
        return _nxn_test_mb(rng, 4, modes, OFFSETS[int(rng.integers(4))], int(rng.choice(_chroma_legal(a, b))))

    return {"mixed_i4": _batch(7, 9, 10, content, seed=3001)}


# ---------------------------------------------------------------------------------------------------------------------
# saturation

def _saturated_mb(luma_hi, chroma_hi):
    """Intra4x4, DC everywhere, one DC level per 4x4 block large enough that the residual (clamped to +-511 by kernel 1)
    drives the block to 0 or 255 whatever the prediction: luma_hi[gy][gx] over the 4x4 grid of blocks, chroma_hi[gy][gx]
    over the 2x2 grid of chroma blocks (both planes)."""
    coeff = np.zeros(384, np.int16)
    for blk in range(16):
        x, y = pred_ref._blk4_xy(blk)
        coeff[blk * 16] = 200 if luma_hi[y // 4][x // 4] else -200
    s = np.array([1 if chroma_hi[k // 2][k % 2] else -1 for k in range(4)])
    hadamard = np.array([[1, 1, 1, 1], [1, -1, 1, -1], [1, 1, -1, -1], [1, -1, -1, 1]])    # f = M c, xform_ref order
    c = hadamard @ (400 * s) // 4                                                          # M^-1 = M / 4
    for p in range(2):
        coeff[256 + 64 * p:320 + 64 * p:16] = c
    return _mb(I4, [2] * 16, chroma=0, coeff=coeff)


def _plane_case():
    """Each 2 x 2 picture: D, B and A built of 0 and 255 blocks so that the bottom line of D and B and the right column of
    A are a step 0...0 / 255...255 (or the reverse) for luma and chroma; the test macroblock at (1, 1) is Intra16x16 and
    chroma plane with no levels.  Signs (H, V) in all four combinations."""
    mbs = []
    tests = []
    for p, (sh, sv) in enumerate([(1, 1), (-1, -1), (1, -1), (-1, 1)] * 2):
        lo_top, lo_left = sh > 0, sv > 0            # the first half of the line is the low one
        corner_lo = lo_top if p < 4 else lo_left     # p[-1,-1] serves H or V: both ways
        d = _saturated_mb([[not corner_lo] * 4] * 4, [[not corner_lo] * 2] * 2)
        bb = _saturated_mb([[gx >= 2 if lo_top else gx < 2 for gx in range(4)]] * 4,
                           [[gx >= 1 if lo_top else gx < 1 for gx in range(2)]] * 2)
        aa = _saturated_mb([[gy >= 2 if lo_left else gy < 2] * 4 for gy in range(4)],
                           [[gy >= 1 if lo_left else gy < 1] * 2 for gy in range(2)])
        test = _i16_test_mb(3, 3)
        mbs += [d, bb, aa, test]
        tests += [(p, 1, 1, (1, 1, 0)) + t for t in test["tests"]]
    return _soa_of(2, 2, mbs), tests


def _flat_case():
    """Every mode of every kind next to neighbours that are all 0 or all 255 (pictures 3 x 2, test macroblock at (1, 1)
    with no levels at all)."""
    recipes = ([(I4, m) for m in range(9)] + [(I8, m) for m in range(9)] + [(I16, m) for m in range(4)])
    mbs, tests = [], []
    p = 0
    for hi in (False, True):
        for k, (kind, mode) in enumerate(recipes):
            flat = _saturated_mb([[hi] * 4] * 4, [[hi] * 2] * 2)
            cm = k % 4
            if kind == I16:
                test = _i16_test_mb(mode, cm)
            else:
                test = _mb(kind, [mode] * 16, chroma=cm)
                test["tests"] = [("i4" if kind == I4 else "i8", blk, mode) for blk in range(16 if kind == I4 else 4)]
                test["tests"].append(("chroma", 0, cm))
            mbs += [flat, flat, flat, flat, test, flat]
            tests += [(p, 1, 1, (1, 1, 1)) + t for t in test["tests"]]
            p += 1
    return _soa_of(3, 2, mbs), tests


def _soa_of(w, h, mbs):
    n = len(mbs)
    return Soa(w, h, n // (w * h), np.array([m["kind"] for m in mbs], np.uint8),
               np.array([m["i16"] for m in mbs], np.uint8), np.array([m["chroma"] for m in mbs], np.uint8),
               np.full(n, QP, np.int8), np.full(n, 0x2F, np.uint8), np.stack([m["modes"] for m in mbs]),
               np.stack([m["coeff"] for m in mbs]))


def _cases():
    return {**_coverage_cases(), **_halo_case(), **_mixed_case()}


SAT_CASES = {"sat_plane": _plane_case, "sat_flat": _flat_case}
CASE_NAMES = sorted(list(COVERAGE_GEOMETRIES) + ["upright_halo_w6", "upright_halo_w13", "mixed_i4"])

_built = {}


def case(name):
    if name not in _built:
        _built.update(_cases())
        _built.update({k: f() for k, f in SAT_CASES.items()})
    return _built[name]


# ---------------------------------------------------------------------------------------------------------------------
# helpers over the decoded pictures

def _tables(soa):
    from oracle import cpu
    return cpu.level_scale(soa.lists4x4, soa.lists8x8[0])


_oracle_cache = {}


def _oracle(name):
    from oracle import cpu
    if name not in _oracle_cache:
        _oracle_cache[name] = cpu.reconstruct(case(name)[0])[0]
    return _oracle_cache[name]


def _planes(soa, yuv):
    W, H = soa.width, soa.height
    return (yuv[:W * H].reshape(H, W).astype(np.int64), yuv[W * H:W * H * 5 // 4].reshape(H // 2, W // 2).astype(np.int64),
            yuv[W * H * 5 // 4:].reshape(H // 2, W // 2).astype(np.int64))


def _neighbour_lines(soa, yuv, test):
    """the samples a test block reads, as lines (left column bottom to top, p[-1,-1], top row left to right)"""
    p, mx, my, (a, b, c), kind, blk, mode = test
    y, cb, cr = _planes(soa, yuv[p])
    if kind == "chroma":
        planes, n, X, Y, xo, yo, ur = (cb, cr), 8, 8 * mx, 8 * my, 0, 0, False
    else:
        n = {"i4": 4, "i8": 8, "i16": 16}[kind]
        xo, yo = (0, 0) if kind == "i16" else _origin(n, blk)
        planes, X, Y = (y,), 16 * mx + xo, 16 * my + yo
        ur = kind != "i16" and _upright(n, blk, a, b, c)
    left, up = xo > 0 or a, yo > 0 or b
    lines = []
    for pl in planes:
        line = list(pl[Y:Y + n, X - 1][::-1]) if left else []
        if left and up:
            line.append(pl[Y - 1, X - 1])
        elif line:
            lines.append(line)
            line = []
        if up:
            line += list(pl[Y - 1, X:X + (2 * n if ur else n)])
        lines.append(line)
    return [ln for ln in lines if len(ln) > 1]


def _equal_neighbour_fraction(name):
    soa, tests = case(name)
    yuv = _oracle(name)
    pairs = equal = 0
    for t in tests:
        for ln in _neighbour_lines(soa, yuv, t):
            ln = np.array(ln)
            pairs += len(ln) - 1
            equal += int(np.sum(ln[1:] == ln[:-1]))
    return equal / pairs


def _texture_clipped_fraction(name):
    soa, _ = case(name)
    y = _oracle(name)[:, :soa.width * soa.height]
    return float(np.mean((y == 0) | (y == 255)))


# ---------------------------------------------------------------------------------------------------------------------
# CPU

def test_legal_combination_count():
    assert len(legal_combinations()) == LEGAL_COMBINATIONS


def test_every_legal_combination_is_a_test_block_several_times():
    """If a builder is edited, coverage cannot shrink without a failure here."""
    counts = Counter()
    for name in CASE_NAMES:
        counts.update(combination(kind, blk, mode, *triple) for _, _, _, triple, kind, blk, mode in case(name)[1])
    legal = legal_combinations()
    assert set(counts) <= legal, sorted(set(counts) - legal)[:10]
    missing = sorted(k for k in legal if counts[k] < REPEATS)
    assert not missing, f"{len(missing)} combinations occur fewer than {REPEATS} times: {missing[:10]}"


def test_upright_cases_cover_every_halo_position():
    """Intra4x4 block 5 and Intra8x8 block 1 in modes 3 and 7, with C available at every column modulo 4 (the position
    inside a halo group of four macroblocks), in a short last group with C and without."""
    seen = set()
    for name in CASE_NAMES:
        soa = case(name)[0]
        w = soa.width_mbs
        for p, mx, my, (a, b, c), kind, blk, mode in case(name)[1]:
            if (kind, blk) in (("i4", 5), ("i8", 1)) and mode in (3, 7) and b:
                short = w % 4 != 0 and mx >= w - w % 4
                seen.add((kind, mode, c, "short" if short else mx % 4))
    for kind in ("i4", "i8"):
        for mode in (3, 7):
            for pos in (0, 1, 2, 3, "short"):
                assert (kind, mode, 1, pos) in seen, (kind, mode, pos)
            assert (kind, mode, 0, "short") in seen, (kind, mode)


def test_mixed_mode_words_pair_dc_with_directional_blocks():
    """In every diagonal step that holds two blocks, the draw has one block DC with both sides while the other is not
    DC, both ways round; and picture-edge DC blocks next to directional ones."""
    soa = case("mixed_i4")[0]
    W = soa.width_mbs
    both_sides, edge = set(), set()
    for addr in range(soa.n_pics * soa.n_mbs):
        if soa.mb_kind[addr] != I4:
            continue
        mx, my = addr % soa.n_mbs % W, addr % soa.n_mbs // W
        a, b = mx > 0, my > 0
        for t in range(2, 8):
            blocks = [(t & 1, t >> 1), ((t & 1) + 2, (t >> 1) - 1)]
            modes, dc_kind = [], []
            for gx, gy in blocks:
                blk = pred_ref._blk4_at(4 * gx, 4 * gy)
                m = int(soa.luma_modes[addr, blk])
                left, up = gx > 0 or a, gy > 0 or b
                modes.append(m)
                dc_kind.append(None if m != 2 else "both" if left and up else "edge")
            for h in (0, 1):
                if dc_kind[h] == "both" and modes[1 - h] != 2:
                    both_sides.add((t, h))
                if dc_kind[h] == "edge" and modes[1 - h] != 2:
                    edge.add((t, h))
    assert both_sides == {(t, h) for t in range(2, 8) for h in (0, 1)}, sorted(both_sides)
    assert {(2, 0), (4, 0), (6, 0), (2, 1), (3, 1)} <= edge, sorted(edge)


@pytest.mark.parametrize("name", CASE_NAMES)
def test_neighbour_lines_are_textured(name):
    """A wrong tap shows only where the sample it reads differs from the right one: few equal neighbours on the lines
    the test blocks read, and few samples at the clip limits."""
    assert _equal_neighbour_fraction(name) < 0.06
    assert _texture_clipped_fraction(name) < 0.01


def test_plane_saturation_reaches_the_limits():
    """|b| = 717 (luma) and |c| = 1355 (chroma) of both signs are reached, and the plane clips on both sides inside one
    macroblock."""
    soa = case("sat_plane")[0]
    yuv = _oracle("sat_plane")
    bs, cs, both = set(), set(), 0
    for p in range(soa.n_pics):
        y, cb, _ = _planes(soa, yuv[p])
        t, l = y[15, 15:32], y[16:32, 15]                   # p[-1..15, -1], p[-1, 0..15]
        H = sum((i + 1) * (t[9 + i] - t[7 - i]) for i in range(8))
        V = sum((i + 1) * (l[8 + i] - (t[0] if i == 7 else l[6 - i])) for i in range(8))
        bs |= {(5 * H + 32) >> 6, (5 * V + 32) >> 6}
        ct, cl = cb[7, 7:16], cb[8:16, 7]
        Hc = sum((i + 1) * (ct[5 + i] - ct[3 - i]) for i in range(4))
        cs.add((34 * Hc + 32) >> 6)
        mb = y[16:32, 16:32]
        both += bool((mb == 0).any() and (mb == 255).any())
    assert {717, -717} <= bs and {1355, -1355} <= cs, (bs, cs)
    assert both >= 2


@pytest.mark.parametrize("name", CASE_NAMES + sorted(SAT_CASES))
def test_pred_ref_matches_oracle_on_edge_cases(name):
    soa = case(name)[0]
    ls4, ls8 = _tables(soa)
    assert np.array_equal(pred_ref.reconstruct(soa, ls4, ls8), _oracle(name))


def test_pred_ref_matches_oracle_and_reference_on_golden_fixtures():
    from helpers import golden_names, load_golden, oracle_reconstruct_with_tables
    for name in golden_names():
        soa, z = load_golden(name)
        want, _ = oracle_reconstruct_with_tables(soa, z["ls4"], z["ls8"])
        got = pred_ref.reconstruct(soa, z["ls4"], z["ls8"])
        assert np.array_equal(got, want), name
        assert np.array_equal(got, z["yuv"]), f"{name}: the reference decoder's own pictures"


@pytest.mark.parametrize("kw", [dict(width_mbs=7, height_mbs=5, profile_idc=100, transform8x8=1, scaling_lists=1, seed=5),
                                dict(width_mbs=1, height_mbs=6, profile_idc=100, transform8x8=1, seed=6),
                                dict(width_mbs=9, height_mbs=2, profile_idc=77, cb_qp_offset=3, seed=7)],
                         ids=["high_7x5", "high_1x6", "main_9x2"])
def test_pred_ref_matches_oracle_on_generated_batches(kw):
    from minivideo_b200 import synth
    from oracle import cpu
    _, soa = synth.generate(3, want_stream=False, **kw)
    ls4, ls8 = _tables(soa)
    assert np.array_equal(pred_ref.reconstruct(soa, ls4, ls8), cpu.reconstruct(soa)[0])


@pytest.mark.parametrize("mutation", pred_ref.MUTATIONS)
def test_every_emulated_mistake_is_caught_by_the_edge_cases(mutation):
    """Each mistake pred_ref can emulate changes the output of at least one edge case: these cases would catch it in a
    kernel."""
    for name in CASE_NAMES + sorted(SAT_CASES):
        soa = case(name)[0]
        ls4, ls8 = _tables(soa)
        if not np.array_equal(pred_ref.reconstruct(soa, ls4, ls8, mutation), _oracle(name)):
            return
    pytest.fail(f"no edge case shows {mutation}")


# ---------------------------------------------------------------------------------------------------------------------
# GPU

def _check_gpu(name):
    from minivideo_b200 import api
    from oracle import cpu
    soa = case(name)[0]
    want_yuv = _oracle(name)
    ls4, ls8 = _tables(soa)
    assert np.array_equal(pred_ref.reconstruct(soa, ls4, ls8), want_yuv), f"{name}: the oracle vs pred_ref"
    want_rgb = {s: cpu.yuv_to_rgb(want_yuv, soa.width, soa.height, s) for s in (1, 2, 4, 8, 16)}
    for mode in (api.PIPELINE_FUSED, api.PIPELINE_SPLIT):
        route = "fused" if mode == api.PIPELINE_FUSED else "split"
        ctx = api.Context(0, soa.width_mbs, soa.height_mbs, soa.n_pics)
        try:
            ctx.set_pipeline_mode(mode)
            ctx.set_sps_from(soa)
            ctx.upload(soa, 0)
            ctx.run(0, soa.n_pics, 1)
            ctx.sync()
            for i in range(soa.n_pics):
                assert np.array_equal(ctx.download_yuv420(i), want_yuv[i]), f"{name} picture {i}: YUV ({route})"
                assert np.array_equal(ctx.download_rgb(i), want_rgb[1][i]), f"{name} picture {i}: RGB ({route} + kernel 3)"
            if mode == api.PIPELINE_SPLIT:
                assert ctx.timing().launches == 3
                continue
            ctx.run_rgb(0, soa.n_pics)
            ctx.sync()
            for i in range(soa.n_pics):
                assert np.array_equal(ctx.download_rgb(i), want_rgb[1][i]), f"{name} picture {i}: RGB (run_rgb)"
            for s in (2, 4, 8, 16):
                ctx.run_thumbs(0, soa.n_pics, s)
                ctx.sync()
                for i in range(soa.n_pics):
                    assert np.array_equal(ctx.download_rgb(i, s), want_rgb[s][i]), f"{name} picture {i}: thumbs 1/{s}"
        finally:
            ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASE_NAMES)
def test_gpu_prediction_edge_cases_match_oracle(name):
    """Tiles -> YUV, tiles -> kernel 3 RGB, run_rgb, run_thumbs at 2, 4, 8, 16 and the split pipeline, byte for byte."""
    _check_gpu(name)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(SAT_CASES))
def test_gpu_prediction_saturation_matches_oracle(name):
    """The same routes where the predictors reach their range limits and the output clips."""
    _check_gpu(name)
