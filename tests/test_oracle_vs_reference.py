"""Check of the oracle (and of the synthetic encoder) against the compiled, unmodified reference in oracle/_ref: live
where oracle/_ref has been built, elsewhere against the results stored in tests/golden/reference_outputs.json (where
they come from: tests/helpers.py, REFERENCE_OUTPUTS)."""
import numpy as np
import pytest

from helpers import reference_output, sha
from oracle import ref

SOA_FIELDS = ("mb_kind", "i16_mode", "chroma_mode", "qp_y", "cbp", "luma_modes", "coeff")

CASES = {
    "cif": (2, dict(config="cif", seed=31)),
    "high_small": (2, dict(width_mbs=7, height_mbs=5, profile_idc=100, transform8x8=1, scaling_lists=1, seed=32,
                           qp_min=0, qp_max=51, cb_qp_offset=-3, cr_qp_offset=5)),
    "main_dense": (1, dict(width_mbs=6, height_mbs=6, profile_idc=77, seed=33, luma_cbp_percent=100, mean_coeffs_x10=150)),
    "sparse": (1, dict(width_mbs=6, height_mbs=6, profile_idc=100, transform8x8=1, seed=34, luma_cbp_percent=5, mean_coeffs_x10=5)),
    "720p": (1, dict(config="720p", seed=35)),
    "1080p": (1, dict(config="1080p", seed=36)),
}


def h(a) -> str:
    """Shape and digest of an array's values (the reference's dump and the generator may store them in other integer
    types)."""
    a = np.asarray(a, np.int32)
    return f"{list(a.shape)} {sha(a)}"


@pytest.mark.parametrize("name", sorted(CASES))
def test_reference_parse_equals_generator_soa_and_oracle_equals_reference(name):
    from minivideo_b200 import synth
    from oracle import cpu
    n, kw = CASES[name]
    stream, soa = synth.generate(n, **kw)

    def live():
        r = ref.decode(stream, n, soa.width, soa.height, want_rgb=True, want_soa=True)
        parsed, ls4, ls8 = ref.parse_soa(r["soa"])
        return dict({f: h(getattr(parsed, f)) for f in SOA_FIELDS}, ls4=h(ls4), ls8=h(ls8), yuv=h(r["yuv"]), rgb=h(r["rgb"]))
    want = reference_output(f"ref_decode {name}", live, ref.available())
    for f in SOA_FIELDS:     # the reference parsed exactly the syntax the encoder meant
        assert h(getattr(soa, f)) == want[f], f
    o4, o8 = cpu.level_scale(soa.lists4x4, soa.lists8x8[0])
    assert h(o4) == want["ls4"] and h(o8) == want["ls8"]
    yuv, _ = cpu.reconstruct(soa)
    assert h(yuv) == want["yuv"]
    assert h(cpu.yuv_to_rgb(yuv, soa.width, soa.height, 1)) == want["rgb"]


@pytest.mark.skipif(not ref.available(), reason="oracle/_ref not built (reference tree not mounted)")
def test_export_tap_equals_the_reference_cli_files():
    """ref_decode's tap (mb_to_ycbcr) writes the same bytes as `mini_thumbnailer -f yuv420`
    (export_idr_yuv420 -> files in the CWD)."""
    from minivideo_b200 import synth
    stream, soa = synth.generate(3, "cif", seed=41)
    a = ref.decode(stream, 3, soa.width, soa.height)["yuv"]
    b = ref.decode_cli(stream, 3, soa.width, soa.height)
    assert np.array_equal(a, b)


def test_cavlc_coverage_every_total_coeff_and_nc_class():
    """Streams dense enough to reach every coeff_token table (nC classes 0-1, 2-3, 4-7, 8+ and
    chroma DC) and TotalCoeff 0..16 round-trip through the reference's CAVLC decoder."""
    from minivideo_b200 import synth
    seen = set()
    for seed, mean in ((51, 20), (52, 80), (53, 160)):
        stream, soa = synth.generate(1, width_mbs=8, height_mbs=6, profile_idc=77, seed=seed, luma_cbp_percent=90,
                                     mean_coeffs_x10=mean, force_kind=0)

        def live():
            r = ref.decode(stream, 1, soa.width, soa.height, want_soa=True)
            parsed, _, _ = ref.parse_soa(r["soa"])
            return h(parsed.coeff)
        assert h(soa.coeff) == reference_output(f"ref_decode cavlc seed {seed}", live, ref.available())
        seen |= set(np.count_nonzero(soa.coeff[:, :256].reshape(-1, 16), axis=1).tolist())
    assert seen == set(range(17))
