"""Shared by the transport-stream and Matroska tests: the four streams tests/test_mp4.py wraps (two of them with
parameter sets that change between pictures), and the check that a container opens to its Annex-B twin."""
import functools

import numpy as np

FIELDS = ("mb_kind", "i16_mode", "chroma_mode", "qp_y", "cbp", "luma_modes", "coeff")
NAMES = ("high", "multi", "multi_size", "two_desc")


@functools.lru_cache(maxsize=None)
def stream(name: str) -> bytes:
    from helpers import paramset_change_stream
    from minivideo_b200 import synth
    if name == "high":
        return synth.generate(6, width_mbs=20, height_mbs=12, profile_idc=100, transform8x8=1, scaling_lists=1,
                              cb_qp_offset=3, cr_qp_offset=-1, seed=611)[0]
    if name == "tiny":          # NAL units below 256 bytes, for 1-byte length fields
        return synth.generate(6, width_mbs=2, height_mbs=1, profile_idc=66, luma_cbp_percent=20, mean_coeffs_x10=5, seed=3)[0]
    if name == "multi":         # three generations of one picture size
        return paramset_change_stream(False)[0]
    if name == "multi_size":    # the second generation changes the picture size too
        return paramset_change_stream(True)[0]
    if name == "two_desc":      # other scaling lists, chroma offsets and picture size half way
        a = synth.generate(3, width_mbs=6, height_mbs=4, profile_idc=100, transform8x8=1, scaling_lists=1,
                           cb_qp_offset=4, cr_qp_offset=-6, seed=613)[0]
        b = synth.generate(4, width_mbs=9, height_mbs=5, profile_idc=100, transform8x8=0, scaling_lists=1,
                           cb_qp_offset=-2, cr_qp_offset=5, seed=614)[0]
        return a.rstrip(b"\x00") + b            # a's last NAL never ends in a zero byte (rbsp_trailing_bits)
    raise KeyError(name)


def assert_same_stream(data: bytes, container: str, es: bytes, all_modes: bool):
    """Stream(data, container) and Stream(es) agree in everything the front end reports, and parse alike."""
    from minivideo_b200 import front
    a, b = front.Stream(data, container), front.Stream(es)
    assert (a.n_idr, a.n_generations) == (b.n_idr, b.n_generations)
    assert b.n_idr > 0
    for g in range(b.n_generations):
        assert bytes(a.generation_info(g)) == bytes(b.generation_info(g)), g
    gens = b.picture_generations()
    assert np.array_equal(a.picture_generations(), gens)
    for n in (1, 2, 3, b.n_idr, b.n_idr + 3):
        for mode in ((0, 1, 2) if all_modes else (0,)):
            assert np.array_equal(a.select_idr(n, mode), b.select_idr(n, mode)), (n, mode)
    for g in range(b.n_generations):
        idx = np.flatnonzero(gens == g).astype(np.int32)
        pa, pb = a.parse(indices=idx), b.parse(indices=idx)
        for f in FIELDS:
            assert np.array_equal(getattr(pa, f), getattr(pb, f)), (g, f)
        ka, kb = a.parse_packed(indices=idx), b.parse_packed(indices=idx)
        assert ka.keys() == kb.keys()
        for k in ka:
            assert np.array_equal(ka[k], kb[k]), (g, k)
