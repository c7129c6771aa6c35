"""Host front end (libmvfront.so): Annex-B / SPS / PPS / slice / CAVLC -> SoA."""
import numpy as np
import pytest

from helpers import golden_names, load_golden
from oracle import ref

FIELDS = ("mb_kind", "i16_mode", "chroma_mode", "qp_y", "cbp", "luma_modes", "coeff")


def same(a, b):
    return all(np.array_equal(getattr(a, f), getattr(b, f)) for f in FIELDS)


@pytest.mark.parametrize("name", golden_names())
def test_front_end_equals_the_reference_parse_on_golden_streams(name):
    """Golden fixtures hold the stream AND the reference's own parsed macroblocks + tables."""
    from minivideo_b200 import front
    want, z = load_golden(name)
    st = front.Stream(z["stream"].tobytes())
    assert (st.info.width_mbs, st.info.height_mbs, st.n_idr) == (want.width_mbs, want.height_mbs, want.n_pics)
    assert (st.info.cb_qp_offset, st.info.cr_qp_offset) == (want.cb_qp_offset, want.cr_qp_offset)
    ls4, ls8 = st.level_scale()
    assert np.array_equal(ls4, z["ls4"]) and np.array_equal(ls8, z["ls8"])
    for threads in (1, 3):
        assert same(st.parse(n_threads=threads), want)


@pytest.mark.parametrize("cfg,n", [("cif", 6), ("720p", 2), ("1080p", 2)])
def test_front_end_equals_generator_soa(cfg, n):
    from minivideo_b200 import front, synth
    stream, soa = synth.generate(n, cfg, seed=77)
    st = front.Stream(stream)
    assert same(st.parse(), soa)
    # sub-ranges and explicit index lists
    assert same(st.parse(first=1, count=n - 1), soa.pictures(1, n - 1))
    assert same(st.parse(indices=[n - 1, 0]), type(soa)(soa.width_mbs, soa.height_mbs, 2,
                *(np.concatenate([getattr(soa.pictures(n - 1, 1), f), getattr(soa.pictures(0, 1), f)]) for f in FIELDS)))


def test_three_byte_start_codes_and_other_nal_types_are_accepted():
    """The reference's ES parser needs 4-byte start codes and knows only 0x65/0x67/0x68
    (esparser.c:78-82); the front end takes the general Annex-B form."""
    from minivideo_b200 import front, synth
    stream, soa = synth.generate(2, "cif", seed=5)
    alt = stream.replace(b"\x00\x00\x00\x01", b"\x00\x00\x01")
    aud = b"\x00\x00\x01\x09\xf0"                       # access unit delimiter
    alt = aud + alt.replace(b"\x00\x00\x01\x65", aud + b"\x00\x00\x01\x25")   # nal_ref_idc 1
    assert same(front.Stream(alt).parse(), soa)


def test_errors_are_reported_not_fatal():
    from minivideo_b200 import front, synth
    with pytest.raises(front.FrontError):
        front.Stream(b"\x00" * 100)
    stream, _ = synth.generate(1, "cif")
    cut = stream[: len(stream) // 2]
    st = front.Stream(cut)
    with pytest.raises(front.FrontError, match="picture 0"):
        st.parse()
    with pytest.raises(front.FrontError, match="out of range"):
        front.Stream(stream).parse(indices=[3])
    cabac = bytearray(stream)
    i = stream.index(b"\x00\x00\x00\x01\x68") + 5
    cabac[i] |= 0x20                                     # ue(0) ue(0) then entropy_coding_mode_flag
    with pytest.raises(front.FrontError, match="CABAC") as e:
        front.Stream(bytes(cabac))
    assert e.value.code == -1


def _interleaved_stream(n, seed=9):
    """n small pictures whose coded sizes alternate between large and tiny."""
    from minivideo_b200 import synth
    kw = dict(width_mbs=4, height_mbs=3, profile_idc=66, seed=seed)
    big, _ = synth.generate(n, luma_cbp_percent=100, mean_coeffs_x10=120, **kw)
    small, _ = synth.generate(n, luma_cbp_percent=0, mean_coeffs_x10=1, **kw)
    def nals(s):
        parts = s[:-64].split(b"\x00\x00\x00\x01")[1:]
        return [b"\x00\x00\x00\x01" + p for p in parts]
    nb, ns = nals(big), nals(small)
    out = nb[0] + nb[1]
    for i in range(n):
        out += (ns if i % 3 == 1 else nb)[2 + i]
    return out + b"\x00" * 64


@pytest.mark.parametrize("mode,flag", [(1, "ordered"), (2, "distributed")])
@pytest.mark.parametrize("n_total,n_want", [(20, 5), (60, 7), (31, 4)])
def test_idr_selection_matches_the_reference_filter(mode, flag, n_total, n_want, tmp_path):
    """mvf_select_idr() vs idr_filtering() (demuxer/filter.c): run the reference CLI with -e ordered /
    distributed and identify which pictures it exported."""
    import subprocess
    from helpers import reference_output
    from minivideo_b200 import front
    stream = _interleaved_stream(n_total)
    st = front.Stream(stream)
    assert st.n_idr == n_total

    def live():
        every = ref.decode(stream, n_total, 64, 48)["yuv"]
        (tmp_path / "in.264").write_bytes(stream)
        subprocess.run([str(ref.MINI_THUMBNAILER), "-i", "in.264", "-f", "yuv420", "-n", str(n_want), "-e", flag],
                       cwd=tmp_path, capture_output=True)
        exported = []
        for i in range(n_want):
            f = tmp_path / f"in_{i}.yuv"
            if not f.exists():
                break
            pic = np.fromfile(f, np.uint8)
            hits = [k for k in range(n_total) if np.array_equal(every[k], pic)]
            assert hits, "reference exported a picture that is not in the stream"
            exported.append(hits[0])
        return exported
    got = reference_output(f"mini_thumbnailer -e {flag} -n {n_want} of {n_total}", live, ref.available())
    mine = st.select_idr(n_want, mode).tolist()
    assert mine[:len(got)] == got and len(mine) >= len(got)
    assert len(got) >= n_want - 1            # the reference may lose the last one (index one past the end)


def test_unfiltered_selection_is_the_first_n():
    from minivideo_b200 import front, synth
    stream, _ = synth.generate(5, width_mbs=2, height_mbs=2, profile_idc=66)
    st = front.Stream(stream)
    assert st.select_idr(3, 0).tolist() == [0, 1, 2]
    assert st.select_idr(9, 0).tolist() == [0, 1, 2, 3, 4]


# ---- parameter sets that change inside the stream (VERDICT r01: "first ones win" was wrong) ------------------------

def _multi():
    import numpy as np
    from helpers import GOLDEN
    return np.load(GOLDEN / "multi_paramsets.npz")


def test_parameter_sets_are_tracked_per_picture():
    """The reference decodes every SPS / PPS where it meets it (h264.c:128-150); later pictures use later tables,
    offsets and pic_init_qp.  The front end reports one parameter generation per distinct (SPS, PPS) pair in force
    and parses each picture with its own."""
    from helpers import paramset_change_stream
    from minivideo_b200 import front
    stream, segs = paramset_change_stream()
    assert stream == _multi()["stream"].tobytes(), "the committed fixture was made from this stream"
    st = front.Stream(stream)
    assert st.n_generations == 3 and list(st.picture_generations()) == [0, 0, 1, 1, 2, 2]
    want = [(26, 0, 0), (33, 5, -4), (21, -3, 2)]
    for g, seg in enumerate(segs):
        info = st.generation_info(g)
        assert (info.pic_init_qp, info.cb_qp_offset, info.cr_qp_offset) == want[g]
        assert (info.n_generations, info.generation) == (3, g)
        assert same(st.parse(first=2 * g, count=2), seg), f"segment {g}: QPs come from this segment's pic_init_qp"
    # generations 1 and 2 share the SPS (same scaling lists), generation 0 has other lists
    l0, l1, l2 = (st.level_scale(st.generation_info(g))[0] for g in range(3))
    assert np.array_equal(l1, l2) and not np.array_equal(l0, l1)
    # one call may span generations of equal picture size: every picture still gets its own parameters
    whole = st.parse()
    for f in FIELDS:
        assert np.array_equal(getattr(whole, f), np.concatenate([getattr(s, f) for s in segs])), f


def test_changing_parameter_sets_reconstruct_like_the_reference():
    """Golden: the reference's own output for the stream above (tests/golden/make_golden.py).  Front end +
    per-generation tables + oracle must reproduce it byte for byte."""
    from helpers import oracle_reconstruct_with_tables
    from minivideo_b200 import front
    from oracle import cpu
    z = _multi()
    st = front.Stream(z["stream"].tobytes())
    gens = st.picture_generations()
    for g in range(st.n_generations):
        idx = [i for i in range(st.n_idr) if gens[i] == g]
        info = st.generation_info(g)
        soa = st.parse(indices=idx)
        yuv, _ = oracle_reconstruct_with_tables(soa, *st.level_scale(info))
        for k, i in enumerate(idx):
            assert np.array_equal(yuv[k], z["yuv"][i]), f"picture {i} (generation {g})"
        assert np.array_equal(cpu.yuv_to_rgb(yuv, soa.width, soa.height, 1), z["rgb"][idx])
    # with the first generation's tables for everything (what round 1 did) pictures 2..5 come out different
    soa = st.parse()
    yuv, _ = oracle_reconstruct_with_tables(soa, *st.level_scale(st.generation_info(0)))
    assert np.array_equal(yuv[:2], z["yuv"][:2]) and not np.array_equal(yuv[2:], z["yuv"][2:])


def test_parameter_set_ids_and_missing_sets():
    """Tables are indexed by id (7.4.1.2.1): a PPS under another id does not disturb pictures that name PPS 0, a
    picture naming a PPS the stream never delivered fails alone, and so does one behind a damaged PPS."""
    from helpers import PAD, split_nals
    from minivideo_b200 import front, synth
    stream, soa = synth.generate(3, width_mbs=4, height_mbs=3, profile_idc=66, seed=17)
    nals = split_nals(stream)
    sps, pps, pics = nals[0], nals[1], nals[2:]
    assert pps[4] == 0x68 and pps[5] & 0x80, "pic_parameter_set_id 0 is coded as the single bit 1"
    # PPS id 1 ('010'), sps id 0 ('1'): the first payload byte 1 1 e b ... becomes 010 1 e b ..: rebuild the bit string
    bits = "".join(f"{b:08b}" for b in pps[5:])
    end = bits.rindex("1")                              # rbsp_stop_one_bit
    body = "010" + bits[1:end] + "1"
    body += "0" * (-len(body) % 8)
    pps1 = pps[:5] + bytes(int(body[i:i + 8], 2) for i in range(0, len(body), 8))
    st = front.Stream(sps + pps + pps1 + b"".join(pics) + PAD)
    assert st.n_generations == 1 and same(st.parse(), soa)
    # no PPS 0 at all: nothing is decodable
    with pytest.raises(front.FrontError, match="PPS 0"):
        front.Stream(sps + pps1 + b"".join(pics) + PAD)
    # PPS 0 arrives after the first picture: picture 0 fails alone (tolerant mode), the others decode
    st = front.Stream(sps + pics[0] + pps + pics[1] + pics[2] + PAD)
    assert list(st.picture_generations()) == [-1, 0, 0]
    with pytest.raises(front.FrontError, match="picture 0"):
        st.parse()
    got = st.parse(tolerant=True)
    assert list(got.status) == [0, 1, 1]
    assert same(got.pictures(1, 2), soa.pictures(1, 2)) and not got.coeff[: soa.n_mbs].any()
