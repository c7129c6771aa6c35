"""kf_recon in the launch regimes production runs in, every picture checked against the oracle.

- Launches with at least 2 * sm_count * KF_WARPS rows, where the row distance switches from KF_GROUP + 1 to
  KF_STAGGER (mvg_api.cu, launch_stages), at the benchmark's 1080p geometry and at a narrow one where the distance is
  clamped to W - 1.
- More than MVG_K2_GROUP (1024) pictures in one launch, so that rows are claimed from several picture groups and the
  last one is short; fused and split pipelines; then a second launch over an overlapping slot range.
- Every row distance the MVG_KF_STAGGER override can set that matters (0 and 1 run rows in lock step), over widths
  on both sides of the group of four and of the distance.
- Geometry changes inside one context, where halo words of the earlier geometry must be rejected by their epoch.

Every batch holds distinct pictures (one generator call), so a picture or row written to the wrong slot shows.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

KF_WARPS = 25           # warps per CTA of kf_recon (mvg_fused.cuh); the row-distance switch is at 2 * sm_count * KF_WARPS rows
HIGH = dict(profile_idc=100, transform8x8=1, scaling_lists=1, cb_qp_offset=3, cr_qp_offset=-2)


def _oracle(soa, i):
    from oracle import cpu
    yuv, _ = cpu.reconstruct(soa.pictures(i, 1))
    return yuv[0]


def _rgb(soa, yuv, scale=1):
    from oracle import cpu
    return cpu.yuv_to_rgb(yuv[None], soa.width, soa.height, scale)[0]


def _context(soa, n_slots):
    from minivideo_b200 import api
    ctx = api.Context(0, soa.width_mbs, soa.height_mbs, n_slots)
    ctx.set_sps_from(soa)
    return ctx


def _check_tiles(ctx, soa, first_slot, what):
    """After run(first_slot, n, 1): YUV from the tiles and RGB from kernel 3 of every picture."""
    for i in range(soa.n_pics):
        want = _oracle(soa, i)
        assert np.array_equal(ctx.download_yuv420(first_slot + i), want), f"{what}: picture {i} YUV"
        assert np.array_equal(ctx.download_rgb(first_slot + i), _rgb(soa, want)), f"{what}: picture {i} RGB (kernel 3)"


def _check_rgb(ctx, soa, first_slot, scale, what):
    """After run_rgb / run_thumbs: the RGB24 of every picture at 1/scale."""
    for i in range(soa.n_pics):
        want = _rgb(soa, _oracle(soa, i), scale)
        assert np.array_equal(ctx.download_rgb(first_slot + i, scale), want), f"{what}: picture {i} RGB 1/{scale}"


def _large_launch(ctx, soa):
    """The three output modes of kf_recon over a launch in the large-launch regime."""
    assert soa.n_pics * soa.height_mbs >= 2 * ctx.sm_count * KF_WARPS, "the launch must be in the large-launch regime"
    ctx.upload(soa, 0)
    ctx.run(0, soa.n_pics, 1)
    ctx.sync()
    assert ctx.timing().launches == 2                   # kf_recon<tiles>, kernel 3
    _check_tiles(ctx, soa, 0, "run")
    ctx.run_rgb(0, soa.n_pics)
    ctx.sync()
    assert ctx.timing().launches == 1                   # kf_recon<rgb>
    _check_rgb(ctx, soa, 0, 1, "run_rgb")
    ctx.run_thumbs(0, soa.n_pics, 4)
    ctx.sync()
    assert ctx.timing().launches == 1                   # kf_recon<thumbnails>
    _check_rgb(ctx, soa, 0, 4, "run_thumbs")


def _sm_count():
    from minivideo_b200 import api
    ctx = api.Context(0, 1, 1, 1)
    try:
        return ctx.sm_count
    finally:
        ctx.close()


def _pics_for_large_launch(height_mbs):
    """Distinct pictures for a launch in the large-launch regime on this GPU, with a margin of 8."""
    return -(-2 * _sm_count() * KF_WARPS // height_mbs) + 8


def test_large_launch_1080p():
    """The benchmark's geometry with enough distinct pictures for the large-launch row distance."""
    from minivideo_b200 import synth
    n = _pics_for_large_launch(68)
    _, soa = synth.generate(n, config="1080p", want_stream=False, seed=0xB200)
    ctx = _context(soa, n)
    try:
        _large_launch(ctx, soa)
    finally:
        ctx.close()


def test_large_launch_narrow():
    """5 x 40 macroblocks: the large-launch row distance (12) is clamped to W - 1 = 4."""
    from minivideo_b200 import synth
    n = _pics_for_large_launch(40)
    _, soa = synth.generate(n, want_stream=False, width_mbs=5, height_mbs=40, seed=0xB201, **HIGH)
    ctx = _context(soa, n)
    try:
        _large_launch(ctx, soa)
    finally:
        ctx.close()


def test_more_than_1024_pictures_and_an_overlapping_relaunch():
    """2 * 1024 + 37 distinct pictures from slot 11: claim groups of 1024 pictures, the last one short.  Fused (tiles and
    RGB) and split pipelines.  Then other content over slots [500, 1700): those pictures must be the new ones, and every
    other slot must still hold the first launch's result."""
    from minivideo_b200 import api, synth
    from oracle import cpu
    first, n = 11, 2 * 1024 + 37
    _, soa = synth.generate(n, want_stream=False, width_mbs=3, height_mbs=4, seed=0xB202, **HIGH)
    want, _ = cpu.reconstruct(soa)
    want_rgb = cpu.yuv_to_rgb(want, soa.width, soa.height, 1)
    ctx = _context(soa, first + n + 40)
    try:
        ctx.upload(soa, first)
        ctx.run(first, n, 1)
        ctx.sync()
        for i in range(n):
            assert np.array_equal(ctx.download_yuv420(first + i), want[i]), f"fused: picture {i} YUV"
            assert np.array_equal(ctx.download_rgb(first + i), want_rgb[i]), f"fused: picture {i} RGB (kernel 3)"
        ctx.run_rgb(first, n)
        ctx.sync()
        for i in range(n):
            assert np.array_equal(ctx.download_rgb(first + i), want_rgb[i]), f"run_rgb: picture {i}"
        ctx.set_pipeline_mode(api.PIPELINE_SPLIT)
        ctx.run(first, n, 1)
        ctx.sync()
        assert ctx.timing().launches == 3
        for i in range(n):
            assert np.array_equal(ctx.download_yuv420(first + i), want[i]), f"split: picture {i} YUV"

        ctx.set_pipeline_mode(api.PIPELINE_FUSED)
        lo, hi = 500, 1700
        _, soa2 = synth.generate(hi - lo, want_stream=False, width_mbs=3, height_mbs=4, seed=0xB203, **HIGH)
        # other levels under the same SPS: the generator draws its scaling lists from the seed, and the context keeps
        # the first batch's tables (the chroma QP offsets are the same by construction)
        soa2.lists4x4, soa2.lists8x8 = soa.lists4x4, soa.lists8x8
        assert (soa2.cb_qp_offset, soa2.cr_qp_offset) == (soa.cb_qp_offset, soa.cr_qp_offset)
        want2, _ = cpu.reconstruct(soa2)
        ctx.upload(soa2, lo)
        ctx.run(lo, hi - lo, 1)
        ctx.sync()
        for slot in range(first, first + n):
            exp = want2[slot - lo] if lo <= slot < hi else want[slot - first]
            assert np.array_equal(ctx.download_yuv420(slot), exp), f"after the overlapping launch: slot {slot}"
    finally:
        ctx.close()


WIDTHS = (1, 2, 4, 5, 8, 9, 13, 33)


@pytest.mark.parametrize("distance", [0, 1, 2, 4, 5, 12, 64])
def test_row_distance_sweep(distance, monkeypatch):
    """MVG_KF_STAGGER (read at context creation) over widths of every residue modulo 4, below and above the group of
    four and the distance, heights 6..9: tiles + YUV, full-size RGB24 and thumbnails at 1/2 and 1/16."""
    from minivideo_b200 import synth
    monkeypatch.setenv("MVG_KF_STAGGER", str(distance))
    for k, w in enumerate(WIDTHS):
        _, soa = synth.generate(3, want_stream=False, width_mbs=w, height_mbs=6 + k % 4, seed=1000 * distance + w, **HIGH)
        ctx = _context(soa, soa.n_pics)
        try:
            ctx.upload(soa, 0)
            what = f"distance {distance}, {w} x {soa.height_mbs}"
            ctx.run(0, soa.n_pics, 1)
            ctx.sync()
            _check_tiles(ctx, soa, 0, what)
            ctx.run_rgb(0, soa.n_pics)
            ctx.sync()
            _check_rgb(ctx, soa, 0, 1, what)
            for scale in (2, 16):
                ctx.run_thumbs(0, soa.n_pics, scale)
                ctx.sync()
                _check_rgb(ctx, soa, 0, scale, what)
        finally:
            ctx.close()


def test_geometry_change_in_one_context():
    """13 x 9, then 12 x 9, then 13 x 9 again in one context: the halo buffer is indexed differently each time and
    only the epoch tells this launch's words from the earlier ones."""
    from minivideo_b200 import api, synth
    n = 6
    soas = [synth.generate(n, want_stream=False, width_mbs=w, height_mbs=9, seed=0xB210 + k, **HIGH)[1]
            for k, w in enumerate((13, 12, 13))]
    ctx = api.Context(0, 13, 9, n)
    try:
        for k, soa in enumerate(soas):
            ctx.set_sps_from(soa)
            ctx.upload(soa, 0)
            ctx.run(0, n, 1)
            ctx.sync()
            _check_tiles(ctx, soa, 0, f"geometry {k}: {soa.width_mbs} x {soa.height_mbs}")
            ctx.run_rgb(0, n)
            ctx.sync()
            _check_rgb(ctx, soa, 0, 1, f"geometry {k}: {soa.width_mbs} x {soa.height_mbs}")
    finally:
        ctx.close()
