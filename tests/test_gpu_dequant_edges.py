"""The transform stage at the extremes the stream generator never emits, on hand-built SoAs: Intra16x16 at every QP
(QP'Y 36 included), one coefficient at every scan position of every block type, levels at the int16 limits, scaling
lists of 1 and 255, chroma QP offsets of +-12 at QP 0 and 51.

Each case is checked three ways: xform_ref.py (numpy, int64 with an explicit 32-bit wrap) against the oracle on the
CPU; the residual of kernel 1 (mvg_download_residual) against both; and the YUV and RGB of the fused kernel kf_recon
(mvg_run, mvg_run_rgb) against the oracle.  Every macroblock is DC-predicted, which needs no neighbour, and the levels
of the YUV cases keep the picture away from 0 and 255, so that a wrong residual inside kf_recon is not hidden by
Clip1(pred + r).
"""
import numpy as np
import pytest

import xform_ref
from minivideo_b200.synth import Soa

W = 19                          # macroblocks per picture row of the hand-built batches
I4, I8, I16 = 0, 1, 2
BASIS_QPS = (0, 5, 6, 23, 24, 35, 36, 51)
_V4_DC = (10, 11, 13, 14, 16, 18)       # normAdjust4x4 at position (0, 0), spec 8.5.9


def _mb(kind, qp, coeff=None):
    return kind, qp, np.zeros(384, np.int16) if coeff is None else coeff


def _soa(mbs, lists4x4=None, lists8x8=None, cb_qp_offset=0, cr_qp_offset=0):
    """A batch of pictures W macroblocks wide holding `mbs` [(kind, qp, coeff[384])] in raster order, padded with empty
    Intra16x16 macroblocks; every prediction mode is DC."""
    h = min(16, -(-len(mbs) // W))
    per = W * h
    n_pics = -(-len(mbs) // per)
    mbs = mbs + [_mb(I16, 26)] * (n_pics * per - len(mbs))
    n = len(mbs)
    soa = Soa(W, h, n_pics, np.array([m[0] for m in mbs], np.uint8), np.full(n, 2, np.uint8), np.zeros(n, np.uint8),
              np.array([m[1] for m in mbs], np.int8), np.full(n, 0x2F, np.uint8), np.full((n, 16), 2, np.uint8),
              np.stack([m[2] for m in mbs]).astype(np.int16), cb_qp_offset=cb_qp_offset, cr_qp_offset=cr_qp_offset)
    if lists4x4 is not None:
        soa.lists4x4 = np.ascontiguousarray(lists4x4, np.uint8)
    if lists8x8 is not None:
        soa.lists8x8 = np.ascontiguousarray(lists8x8, np.uint8)
    return soa


# ---------------------------------------------------------------------------------------------------------------------
# cases

def _i16_dc_level(qp):
    """An Intra16x16 DC level whose residual is about 8 in every block: dcY ~ c * LS * 2^(qP/6) / 64, r ~ dcY / 64
    (DC prediction carries every macroblock's offset on to its neighbours: larger values drift into the clip limits)."""
    return max(1, round(8 * 4096 / (16 * _V4_DC[qp % 6] * 2 ** (qp // 6))))


def i16_dc_mbs(qps=range(52), level=None):
    """One macroblock per (QP, Hadamard position): a single luma DC level of alternating sign."""
    out = []
    for qp in qps:
        for blk in range(16):
            c = np.zeros(384, np.int16)
            v = _i16_dc_level(qp) if level is None else level
            c[blk * 16] = v if (blk + qp) % 2 == 0 or level is not None else -v
            out.append(_mb(I16, qp, c))
    return out


def mid_level(qp):
    """A level of a few bits whose 4x4 residual stays near +-16 (d ~ c * 16 * 16 * 2^(qP/6) / 16, r ~ d / 64)."""
    return max(2, round(64 / 2 ** (qp // 6)))


def basis_mbs(qp, level, alternate=True):
    """One non-zero level per block, so that over the macroblocks of the case every block of every type takes every
    scan position: Intra4x4 (16 macroblocks), Intra8x8 (64), Intra16x16 AC positions 1..15 (15), chroma DC (4), chroma
    AC positions 1..15 (15).  With `alternate`, signs alternate between blocks."""
    out = []
    neg = -level if alternate else level
    for m in range(16):
        c = np.zeros(384, np.int16)
        for blk in range(16):
            c[blk * 16 + (m + blk) % 16] = level if blk % 2 == 0 else neg
        out.append(_mb(I4, qp, c))
    for m in range(64):
        c = np.zeros(384, np.int16)
        for b8 in range(4):
            c[b8 * 64 + (m + 16 * b8) % 64] = level if b8 % 2 == 0 else neg
        out.append(_mb(I8, qp, c))
    for m in range(15):
        c = np.zeros(384, np.int16)
        for blk in range(16):
            c[blk * 16 + 1 + (m + blk) % 15] = level if blk % 2 == 0 else neg
        out.append(_mb(I16, qp, c))
    for m in range(4):
        c = np.zeros(384, np.int16)
        c[256 + m * 16] = level
        c[320 + (m + 1) % 4 * 16] = neg
        out.append(_mb(I16, qp, c))
    for m in range(15):
        c = np.zeros(384, np.int16)
        for blk in range(8):
            c[256 + blk * 16 + 1 + (m + blk) % 15] = level if blk % 2 == 0 else neg
        out.append(_mb(I16, qp, c))
    return out


def basis_soa():
    mbs = []
    for qp in BASIS_QPS:
        for level in (1, -1, mid_level(qp), -mid_level(qp)):
            mbs += basis_mbs(qp, level)
    return _soa(mbs)


def extreme_soa():
    """Single levels at the int16 limits at QP 51 in every scan position: residual only."""
    mbs = []
    for level in (32767, -32767, -32768):
        mbs += basis_mbs(51, level, alternate=False) + i16_dc_mbs([51], level)
    return _soa(mbs)


def dense_extreme_soa(lists=None):
    """Every level of the macroblock at the int16 limits (random signs) at QP 24..51: the dequantised values and the
    sums of the inverse transforms leave the int32 range, where the decoding process wraps modulo 2^32."""
    rng = np.random.default_rng(51)
    mbs = []
    for qp in (24, 36, 42, 47, 51):
        for kind in (I4, I8, I16):
            for _ in range(4):
                mbs.append(_mb(kind, qp, rng.choice(np.array([32767, -32767, -32768], np.int16), 384)))
    return _soa(mbs, lists4x4=lists and np.full((6, 16), lists), lists8x8=lists and np.full((2, 64), lists))


def dc_rounding_soa():
    """DC-only blocks whose level is non-zero but whose residual rounds to 0 (and the neighbours of that boundary):
    quant4x4 of +-1 at QP 0..5 gives d = +-10..+-18, (d + 32) >> 6 = 0; Intra16x16 and chroma DC levels of +-1 at low
    QP come out of their DC transforms just as small."""
    mbs = []
    for qp in range(0, 18):
        for level in (1, -1, 2, -2, 3, -3):
            c = np.zeros(384, np.int16)
            for blk in range(16):
                c[blk * 16] = level
            c[256:384:16] = level
            mbs.append(_mb(I4, qp, c))
            c16 = np.zeros(384, np.int16)
            c16[0] = level
            c16[256] = level
            c16[320 + 48] = -level
            mbs.append(_mb(I16, qp, c16))
    return _soa(mbs)


LIST_CASES = {
    "all_1": lambda rng: (np.ones((6, 16)), np.ones((2, 64))),
    "all_255": lambda rng: (np.full((6, 16), 255), np.full((2, 64), 255)),
    "random": lambda rng: (rng.integers(1, 256, (6, 16)), rng.integers(1, 256, (2, 64))),
}


def lists_soa(name):
    """Random levels in every macroblock type at every QP 0..51, with the scaling lists of `name`."""
    rng = np.random.default_rng(sum(map(ord, name)))
    l4, l8 = LIST_CASES[name](rng)
    mbs = []
    for qp in range(52):
        for kind in (I4, I8, I16):
            c = np.where(rng.random(384) < 0.3, rng.integers(-40, 41, 384), 0).astype(np.int16)
            mbs.append(_mb(kind, qp, c))
    return _soa(mbs, lists4x4=l4, lists8x8=l8)


OFFSETS = [(-12, 12), (12, -12)]


def offsets_soa(cb, cr):
    """Chroma DC and AC levels at QP'Y 0, 1, 50, 51 with chroma QP offsets of +-12: both clamps of Table 8-15."""
    mbs = []
    for qp in (0, 1, 50, 51):
        dc = max(1, round(32 / 2 ** (qp // 6)))
        for m in range(16):
            c = np.zeros(384, np.int16)
            for blk in range(8):
                c[256 + blk * 16] = dc * (2 * ((m + blk) % 2) - 1) * (1 + (m + blk) % 3)
                c[256 + blk * 16 + 1 + (m + blk) % 15] = 1 if blk % 2 else -1
            mbs.append(_mb((I4, I8, I16)[m % 3], qp, c))
    return _soa(mbs, cb_qp_offset=cb, cr_qp_offset=cr)


YUV_CASES = {
    "i16_dc_all_qps": lambda: _soa(i16_dc_mbs()),
    "basis": basis_soa,
    "dc_rounding": dc_rounding_soa,
    **{f"chroma_offsets_{cb}_{cr}": (lambda cb=cb, cr=cr: offsets_soa(cb, cr)) for cb, cr in OFFSETS},
}
RESIDUAL_CASES = {
    "extreme_levels": extreme_soa,
    "extreme_dense": dense_extreme_soa,
    "extreme_dense_lists_255": lambda: dense_extreme_soa(255),
    **{f"lists_{k}": (lambda k=k: lists_soa(k)) for k in LIST_CASES},
}


def _tables(soa):
    from oracle import cpu
    return cpu.level_scale(soa.lists4x4, soa.lists8x8[0])


def _clipped_fraction(soa, yuv):
    y = yuv[:, :soa.width * soa.height]
    return float(np.mean((y == 0) | (y == 255)))


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the numpy reference against the oracle

@pytest.mark.parametrize("name", sorted(YUV_CASES) + sorted(RESIDUAL_CASES))
def test_xform_ref_matches_oracle_on_edge_cases(name):
    from oracle import cpu
    soa = {**YUV_CASES, **RESIDUAL_CASES}[name]()
    ls4, ls8 = _tables(soa)
    _, want = cpu.reconstruct(soa, want_residual=True)
    assert np.array_equal(xform_ref.residual(soa, ls4, ls8), want)


def test_xform_ref_matches_oracle_on_golden_fixtures():
    from helpers import golden_names, load_golden, oracle_reconstruct_with_tables
    for name in golden_names():
        soa, z = load_golden(name)
        _, want = oracle_reconstruct_with_tables(soa, z["ls4"], z["ls8"], want_residual=True)
        assert np.array_equal(xform_ref.residual(soa, z["ls4"], z["ls8"]), want), name


@pytest.mark.parametrize("name", sorted(LIST_CASES))
def test_level_scale_restatement_matches_oracle(name):
    from oracle import cpu
    soa = lists_soa(name)
    want = cpu.level_scale(soa.lists4x4, soa.lists8x8[0])
    got = xform_ref.level_scale(soa.lists4x4, soa.lists8x8[0])
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])


def test_chroma_qp_restatement_matches_oracle():
    from oracle import cpu
    L = cpu.lib()
    for qp in range(52):
        for off in range(-12, 13):
            assert int(xform_ref.chroma_qp(qp, off)) == L.oracle_chroma_qp(qp, off), (qp, off)


@pytest.mark.parametrize("name", sorted(YUV_CASES))
def test_yuv_cases_stay_away_from_the_clip_limits(name):
    """The YUV comparisons below observe the residual, not only Clip1: under 1 % of the luma samples are 0 or 255."""
    from oracle import cpu
    soa = YUV_CASES[name]()
    yuv, _ = cpu.reconstruct(soa)
    assert _clipped_fraction(soa, yuv) < 0.01


# ---------------------------------------------------------------------------------------------------------------------
# GPU

def _gpu_residual(ctx, soa):
    return np.concatenate([ctx.download_residual(i) for i in range(soa.n_pics)])


def _context(soa):
    from minivideo_b200 import api
    ctx = api.Context(0, soa.width_mbs, soa.height_mbs, soa.n_pics)
    ctx.set_sps_from(soa)
    ctx.upload(soa, 0)
    return ctx


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(YUV_CASES))
def test_gpu_edge_cases_match_oracle(name):
    """Residual of kernel 1 against the oracle and the numpy reference; YUV (tiles) and RGB (tiles + kernel 3, and
    kf_recon straight to RGB24) of the fused kernel against the oracle."""
    from oracle import cpu
    soa = YUV_CASES[name]()
    want_yuv, want_res = cpu.reconstruct(soa, want_residual=True)
    assert _clipped_fraction(soa, want_yuv) < 0.01
    want_rgb = cpu.yuv_to_rgb(want_yuv, soa.width, soa.height, 1)
    ls4, ls8 = _tables(soa)
    ctx = _context(soa)
    try:
        ctx.run(0, soa.n_pics, 1)
        ctx.sync()
        for i in range(soa.n_pics):
            assert np.array_equal(ctx.download_yuv420(i), want_yuv[i]), f"{name} picture {i}: YUV (kf_recon tiles)"
            assert np.array_equal(ctx.download_rgb(i), want_rgb[i]), f"{name} picture {i}: RGB (tiles + kernel 3)"
        ctx.run_rgb(0, soa.n_pics)
        ctx.sync()
        for i in range(soa.n_pics):
            assert np.array_equal(ctx.download_rgb(i), want_rgb[i]), f"{name} picture {i}: RGB (kf_recon direct)"
        res = _gpu_residual(ctx, soa)
    finally:
        ctx.close()
    assert np.array_equal(res, want_res), f"{name}: kernel 1 residual vs the oracle"
    assert np.array_equal(res, xform_ref.residual(soa, ls4, ls8)), f"{name}: kernel 1 residual vs the numpy reference"


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(RESIDUAL_CASES))
def test_gpu_residual_edge_cases_match_oracle(name):
    """Levels at the int16 limits and scaling lists of 1 and 255 (every QP 0..51): the residual of kernel 1 against
    the oracle and the numpy reference, and the LevelScale tables of the library against the oracle's."""
    from minivideo_b200 import api
    from oracle import cpu
    soa = RESIDUAL_CASES[name]()
    ls4, ls8 = _tables(soa)
    g4, g8 = api.build_level_scale(soa.lists4x4, soa.lists8x8[0])
    assert np.array_equal(g4, ls4) and np.array_equal(g8, ls8)
    _, want = cpu.reconstruct(soa, want_residual=True)
    ctx = _context(soa)
    try:
        res = _gpu_residual(ctx, soa)
    finally:
        ctx.close()
    assert np.array_equal(res, want)
    assert np.array_equal(res, xform_ref.residual(soa, ls4, ls8))
