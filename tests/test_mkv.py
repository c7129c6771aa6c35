"""Matroska / WebM input of the host front end (mvf_open_mkv): a Matroska file holding the NAL units of an Annex-B
stream opens to the same stream -- pictures, parameter generations, selection and parsed macroblocks -- as the
Annex-B stream, for every variant tests/mkv_mux.py writes; damaged files are refused with a code and a message."""
import os

import numpy as np
import pytest

from container_cases import FIELDS, NAMES, assert_same_stream, stream
from mkv_mux import es_twin, mux
from mp4_mux import nal_units

# (knobs, whether every frame is one IDR NAL behind a 4-byte length field -- only then does the frame size equal the
# Annex-B distance, and ordered / distributed selection can be compared -- for a stream whose parameter sets all go
# into CodecPrivate)
KNOBS = {
    "plain": (dict(), True),
    "length2": (dict(length_size=2), False),
    "segment_unknown": (dict(segment_unknown=True), True),
    "cluster_unknown": (dict(cluster_unknown=True, per_cluster=3), True),
    "both_unknown": (dict(segment_unknown=True, cluster_unknown=True, seek_cues_void=True), True),
    "block_group": (dict(block_group=True), True),
    "xiph_lacing": (dict(lacing="xiph", per_block=3), True),
    "ebml_lacing": (dict(lacing="ebml", per_block=4, cluster_unknown=True), True),
    "fixed_lacing": (dict(lacing="fixed", per_block=2), False),
    "block_group_laced": (dict(block_group=True, lacing="ebml", per_block=2), True),
    "audio_first": (dict(audio_first=True), True),
    "seek_cues_void": (dict(seek_cues_void=True), True),
    "in_band": (dict(in_band=True), False),
}


@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("knob", sorted(KNOBS))
def test_mkv_opens_to_the_annexb_stream(knob, name):
    kw, all_modes = KNOBS[knob]
    es = stream(name)
    assert_same_stream(mux(es, **kw), "mkv", es_twin(es), all_modes and name == "high")


@pytest.mark.parametrize("kw", [dict(length_size=1), dict(length_size=1, lacing="xiph", per_block=3, block_group=True)],
                         ids=["length1", "length1_xiph_group"])
def test_one_byte_length_fields(kw):
    es = stream("tiny")
    assert_same_stream(mux(es, **kw), "mkv", es_twin(es), False)


def test_cif_baseline_and_generator_soa():
    from minivideo_b200 import front, synth
    es, soa = synth.generate(5, "cif", seed=612)
    got = front.Stream(mux(es, lacing="xiph", per_block=2), "mkv").parse()
    for f in FIELDS:
        assert np.array_equal(getattr(got, f), getattr(soa, f)), f


def test_a_damaged_frame_skips_only_its_own_nal_units():
    from minivideo_b200 import synth
    es = stream("high")
    other = nal_units(synth.generate(1, width_mbs=7, height_mbs=3, profile_idc=66, seed=615)[0])
    for k in (0, 2, 5):
        for kw in (dict(), dict(lacing="ebml", per_block=3)):
            data = mux(es, damaged_frame=(k, [other[0], other[2]]), **kw)
            assert_same_stream(data, "mkv", es_twin(es), not kw)


def test_bytes_of_another_container_are_a_value_error():
    """Annex-B bytes handed to a container opener are refused by it, with its message, as an OpenError: a FrontError
    and a ValueError."""
    from minivideo_b200 import front
    es = stream("high")
    for container, msg in (("mp4", "overlapping box at offset 0"), ("ts", "no sync bytes"), ("mkv", "no EBML header")):
        with pytest.raises(front.OpenError, match=msg) as e:
            front.Stream(es, container)
        assert isinstance(e.value, ValueError) and isinstance(e.value, front.FrontError) and e.value.code == 0


# ---- refusals ------------------------------------------------------------------------------------------------------

def refusals():
    es = stream("high")
    yield "hevc", mux(es, codec_id=b"V_MPEGH/ISO/HEVC"), -1, "holds V_MPEGH/ISO/HEVC, not H.264"
    yield "vp9", mux(es, codec_id=b"V_VP9"), -1, "holds V_VP9, not H.264"
    yield "webm_vp9", mux(es, codec_id=b"V_VP9", doctype=b"webm"), -1, "holds V_VP9"
    yield "vfw", mux(es, codec_id=b"V_MS/VFW/FOURCC"), -1, "V_MS/VFW/FOURCC"
    yield "content_encodings", mux(es, content_encodings=True), -1, "ContentEncodings"
    yield "no_video", mux(es, video_track=False, audio_first=True), -1, "no video track"
    yield "webm_audio_only", mux(es, video_track=False, audio_first=True, doctype=b"webm"), -1, "WebM file without an H.264"
    yield "no_codec_private", mux(es, codec_private=False), 0, "no CodecPrivate"
    base = mux(es)
    priv = base.index(b"\x63\xa2") + 2
    priv += 9 - base[priv].bit_length()                 # the avcC starts behind the size
    b = bytearray(base)
    b[priv + 4] = 0xFE
    yield "length_size_3", bytes(b), 0, "lengthSizeMinusOne 2 is invalid"
    b = bytearray(base)
    b[priv + 6:priv + 8] = b"\xff\xff"
    yield "codec_private_sps_overrun", bytes(b), 0, "avcC parameter set runs past its CodecPrivate"
    yield "no_ebml_header", base[4:], 0, "no EBML header"
    yield "truncated", base[:-50], 0, "damaged"
    seg = base.index(b"\x18\x53\x80\x67")
    b = bytearray(base)
    b[seg + 4:seg + 12] = (len(base) * 2 | 1 << 56).to_bytes(8, "big")
    yield "segment_past_file", bytes(b), 0, "damaged element|no Segment"
    laced = mux(es, lacing="xiph", per_block=3)
    blk = laced.index(b"\xa3", laced.index(b"\x1f\x43\xb6\x75") + 4)
    b = bytearray(laced)
    hdr = blk + 1 + 9 - b[blk + 1].bit_length()         # behind the SimpleBlock size
    b[hdr + 4] = 0xFF                                   # 256 frames: the Xiph sizes run out
    yield "lace_overrun", bytes(b), 0, "lace sizes overrun their block"
    fixed = mux(es, lacing="fixed", per_block=2)
    blk = fixed.index(b"\xa3", fixed.index(b"\x1f\x43\xb6\x75") + 4)
    b = bytearray(fixed)
    w = 9 - b[blk + 1].bit_length()
    hdr = blk + 1 + w
    laced_bytes = int.from_bytes(b[blk + 1:hdr], "big") - (1 << (7 * w)) - 5      # behind track, timecode, flags, count
    b[hdr + 4] = next(n for n in range(2, 255) if laced_bytes % (n + 1))     # a frame count that does not divide them
    yield "fixed_lace_uneven", bytes(b), 0, "lace sizes overrun their block"


@pytest.mark.parametrize("case", list(refusals()), ids=lambda c: c[0])
def test_damaged_or_unsupported_files_are_refused(case):
    from minivideo_b200 import front
    _, data, code, msg = case
    with pytest.raises(front.FrontError, match=msg) as e:
        front.Stream(data, "mkv")
    assert e.value.code == code, str(e.value)


# ---- a large file ------------------------------------------------------------------------------------------------

def _rss() -> int:
    with open("/proc/self/statm") as f:
        return int(f.read().split()[1]) * os.sysconf("SC_PAGE_SIZE")


def test_a_1000_picture_1080p_file_is_indexed_in_place():
    """About 1 GB of 1080p IDR pictures in unknown-size Clusters: the Matroska file opens to the Annex-B stream's
    pictures and selection, and opening it copies no media data."""
    from helpers import split_nals
    from minivideo_b200 import front, synth
    s, _ = synth.generate(40, "1080p", want_soa=False, luma_cbp_percent=100, mean_coeffs_x10=220, level_scale_x10=30, seed=616)
    nals = split_nals(s)
    es = b"".join(nals[:2] + nals[2:] * 25) + bytes(64)
    del s, nals
    mkv = mux(es, cluster_unknown=True, per_cluster=25)
    assert len(mkv) > 900 << 20
    before = _rss()
    a = front.Stream(mkv, "mkv")
    grown = _rss() - before
    assert grown < 64 << 20, grown
    b = front.Stream(es_twin(es))
    assert a.n_idr == b.n_idr == 1000
    for mode in (0, 1, 2):
        for n in (1, 9, 100, 1000):
            assert np.array_equal(a.select_idr(n, mode), b.select_idr(n, mode)), (n, mode)
    idx = np.array([0, 517, 999], np.int32)
    pa, pb = a.parse(indices=idx), b.parse(indices=idx)
    for f in FIELDS:
        assert np.array_equal(getattr(pa, f), getattr(pb, f)), f
