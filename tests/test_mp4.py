"""MP4 / QuickTime input of the host front end (mvf_open_mp4): an MP4 file holding the NAL units of an Annex-B stream
opens to the same stream -- pictures, parameter generations, selection and parsed macroblocks -- as the Annex-B
stream itself, for every container variant tests/mp4_mux.py writes; damaged files are refused with a code and a
message."""
import functools
import os
import struct

import numpy as np
import pytest

from mp4_mux import es_twin, mux, nal_units

FIELDS = ("mb_kind", "i16_mode", "chroma_mode", "qp_y", "cbp", "luma_modes", "coeff")


@functools.lru_cache(maxsize=None)
def stream(name: str) -> bytes:
    from helpers import paramset_change_stream
    from minivideo_b200 import synth
    if name == "high":
        return synth.generate(6, width_mbs=20, height_mbs=12, profile_idc=100, transform8x8=1, scaling_lists=1,
                              cb_qp_offset=3, cr_qp_offset=-1, seed=611)[0]
    if name == "cif":
        return synth.generate(5, "cif", seed=612)[0]
    if name == "tiny":          # NAL units below 256 bytes, for 1-byte length fields
        return synth.generate(6, width_mbs=2, height_mbs=1, profile_idc=66, luma_cbp_percent=20, mean_coeffs_x10=5, seed=3)[0]
    if name == "multi":         # the multi_paramsets fixture: three generations of one picture size
        return paramset_change_stream(False)[0]
    if name == "multi_size":    # the second generation changes the picture size too
        return paramset_change_stream(True)[0]
    if name == "two_desc":      # two sample descriptions: other scaling lists, chroma offsets and picture size
        a = synth.generate(3, width_mbs=6, height_mbs=4, profile_idc=100, transform8x8=1, scaling_lists=1,
                           cb_qp_offset=4, cr_qp_offset=-6, seed=613)[0]
        b = synth.generate(4, width_mbs=9, height_mbs=5, profile_idc=100, transform8x8=0, scaling_lists=1,
                           cb_qp_offset=-2, cr_qp_offset=5, seed=614)[0]
        return a.rstrip(b"\x00") + b            # a's last NAL never ends in a zero byte (rbsp_trailing_bits)
    raise KeyError(name)


def assert_same_stream(mp4: bytes, es: bytes, all_modes: bool):
    """Stream(mp4, "mp4") and Stream(es) agree in everything the front end reports, and parse alike."""
    from minivideo_b200 import front
    a, b = front.Stream(mp4, "mp4"), front.Stream(es)
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


# (knobs, whether the sample size equals the Annex-B distance of every IDR picture: one IDR NAL per sync sample
# behind a 4-byte length field -- only then can ordered / distributed selection be compared)
KNOBS = {
    "plain": (dict(), True),
    "length2": (dict(length_size=2), False),
    "co64": (dict(co64=True), True),
    "chunks": (dict(chunk_pattern=(2, 1, 3, 3, 1, 4), chunk_gaps=True), True),
    "moov_last": (dict(moov_first=False), True),
    "largesize_mdat": (dict(largesize_mdat=True), True),
    "largesize_mdat_moov_last": (dict(largesize_mdat=True, moov_first=False), True),
    "audio_first": (dict(audio_first=True, chunk_pattern=(2,)), True),
    "junk_non_sync": (dict(junk_samples=2), True),
    "aud_sei": (dict(aud_sei=True), False),
    "avc3": (dict(avc3=True), False),
    "no_high_tail": (dict(high_tail=False), True),
    "constant_size": (dict(constant_size=True), False),
    "no_ftyp": (dict(brand=None), True),
    "qt_brand": (dict(brand=b"qt  ", chunk_pattern=(3,), co64=True), True),
}


@pytest.mark.parametrize("name", ["high", "multi", "multi_size", "two_desc"])
@pytest.mark.parametrize("knob", sorted(KNOBS))
def test_mp4_opens_to_the_annexb_stream(knob, name):
    kw, all_modes = KNOBS[knob]
    es = stream(name)
    assert_same_stream(mux(es, **kw), es_twin(es), all_modes)


@pytest.mark.parametrize("kw", [dict(length_size=1), dict(length_size=1, junk_samples=1, chunk_pattern=(3,))],
                         ids=["length1", "length1_junk"])
def test_one_byte_length_fields(kw):
    es = stream("tiny")
    assert_same_stream(mux(es, **kw), es_twin(es), False)


def test_cif_baseline_and_generator_soa():
    from minivideo_b200 import front, synth
    es, soa = synth.generate(5, "cif", seed=612)
    got = front.Stream(mux(es, chunk_pattern=(2,)), "mp4").parse()
    for f in FIELDS:
        assert np.array_equal(getattr(got, f), getattr(soa, f)), f


def test_a_damaged_sample_skips_only_its_own_nal_units():
    """A sample whose last length field runs past its end: none of its NAL units count -- not the valid SPS in front
    (which would change the picture size of everything after it) and not the IDR picture -- and every other sample
    still does."""
    from minivideo_b200 import synth
    es = stream("high")
    other = nal_units(synth.generate(1, width_mbs=7, height_mbs=3, profile_idc=66, seed=615)[0])
    for k in (0, 2, 5):
        for junk in (0, 1):
            mp4 = mux(es, junk_samples=junk, damaged_sample=(k * (junk + 1), [other[0], other[2]]))
            assert_same_stream(mp4, es_twin(es), True)


def test_container_is_checked():
    from minivideo_b200 import front
    with pytest.raises(ValueError):
        front.Stream(stream("high"), "mkv")
    with pytest.raises(front.FrontError, match="overlapping box at offset 0") as e:
        front.Stream(stream("high"), "mp4")         # Annex-B bytes are no MP4 file
    assert e.value.code == 0


# ---- refusals -------------------------------------------------------------------------------------------------

CONTAINERS = {b"moov", b"trak", b"mdia", b"minf", b"stbl", b"dinf"}


def boxes(data: bytes, start: int = 0, end: int | None = None, path: str = "") -> dict:
    """{"moov/trak/mdia/...": [header offset, ...]} of every box in the container tree (sample entries not included)."""
    out, pos, end = {}, start, len(data) if end is None else end
    while pos < end:
        size, kind = struct.unpack(">I4s", data[pos:pos + 8])
        hdr = 8
        if size == 1:
            size, hdr = struct.unpack(">Q", data[pos + 8:pos + 16])[0], 16
        p = path + kind.decode("latin-1")
        out.setdefault(p, []).append(pos)
        if kind in CONTAINERS:
            for k, v in boxes(data, pos + hdr, pos + size, p + "/").items():
                out.setdefault(k, []).extend(v)
        pos += size
    return out


STBL = "moov/trak/mdia/minf/stbl/"


def patch(data: bytes, off: int, value: int, fmt: str = ">I") -> bytes:
    b = bytearray(data)
    struct.pack_into(fmt, b, off, value)
    return bytes(b)


def rename(data: bytes, old: bytes, new: bytes, start: int = 0) -> bytes:
    """The first four-character code `old` from offset `start` on becomes `new`."""
    i = data.index(old, start)
    return data[:i] + new + data[i + 4:]


def refusals():
    """(id, mp4 bytes, return code, message) for one case of every way mvf_open_mp4 refuses a file."""
    es = stream("high")
    base = mux(es, moov_first=False, chunk_pattern=(2, 1, 3))
    bx = boxes(base)
    moov = bx["moov"][0]
    stsz, stsc, stco = bx[STBL + "stsz"][0], bx[STBL + "stsc"][0], bx[STBL + "stco"][0]
    stsd = bx[STBL + "stsd"][0]
    n_samples = struct.unpack(">I", base[stsz + 16:stsz + 20])[0]
    mvex = struct.pack(">I4s", 8, b"mvex")
    yield "moof", base + struct.pack(">I4s", 8, b"moof"), -1, "fragmented file \\(moof\\)"
    yield "mvex", patch(base, moov, len(base) - moov + 8) + mvex, -1, "fragmented file \\(mvex\\)"
    yield "hvc1", rename(base, b"avc1", b"hvc1", stsd), -1, "'hvc1', not H.264"
    yield "encv", rename(base, b"avc1", b"encv", stsd), -1, "'encv', not H.264"
    yield "no_video", rename(base, b"vide", b"soun"), -1, "no video track"
    audio_only = mux(es, audio_first=True)
    yield "audio_only", rename(audio_only, b"vide", b"text"), -1, "no video track"
    multi = mux(stream("multi"))
    first_entry = multi.index(b"avc1", boxes(multi)[STBL + "stsd"][0])
    yield "second_description_not_avc", rename(multi, b"avc1", b"hvc1", first_entry + 4), -1, "sample description 2 is 'hvc1'"
    yield "no_moov", base[:moov], 0, "no moov box"
    yield "truncated_moov", base[:-9], 0, "truncated or overlapping box at offset"
    yield "truncated_mdat", mux(es)[:-100], 0, "truncated or overlapping box at offset"
    yield "size_below_header", patch(base, stsz, 7), 0, "truncated or overlapping box"
    yield "size_past_parent", patch(base, stsz, len(base) - stsz + 1), 0, "truncated or overlapping box"
    yield "largesize_below_header", patch(patch(base, moov, 1), moov + 8, 12, ">Q"), 0, "truncated or overlapping box"
    yield "stsz_count_overflow", patch(base, stsz + 16, 0xFFFFFFFF), 0, "stsz sample count 4294967295 exceeds its box"
    yield "stsz_constant_count_too_large", patch(patch(base, stsz + 12, 5), stsz + 16, 0xFFFFFFF), 0, "exceeds the file size"
    yield "stsc_count_overflow", patch(base, stsc + 12, 0xFFFFFFFF), 0, "stsc entry count 4294967295 exceeds its box"
    yield "stco_count_overflow", patch(base, stco + 12, 0x40000000), 0, "chunk offset count 1073741824 exceeds its box"
    yield "stsd_count_overflow", patch(base, stsd + 12, 0xFFFFFFFF), 0, "stsd entry count 4294967295 exceeds its box"
    yield "stsc_first_chunk_not_1", patch(base, stsc + 16, 2), 0, "first_chunk 2"
    yield "stsc_first_chunk_repeats", patch(base, stsc + 16 + 12, 1), 0, "stsc entry 1: first_chunk 1"
    yield "stsc_description_0", patch(base, stsc + 16 + 8, 0), 0, "names sample description 0 of 1"
    yield "stsc_description_2", patch(base, stsc + 16 + 8, 2), 0, "names sample description 2 of 1"
    yield "chunk_outside_file", patch(base, stco + 16, len(base) + 1), 0, "chunk 1 lies outside the file"
    last = stsz + 20 + 4 * (n_samples - 1)
    yield "sample_outside_file", patch(base, last, len(base)), 0, f"sample {n_samples} lies outside the file"
    yield "stsz_fewer_than_stsc", patch(base, stsz + 16, n_samples - 1), 0, "stsc describes more samples"
    yield "stsz_more_than_stsc", patch(base, stsz + 16, n_samples + 1), 0, "exceeds its box|stsc describes fewer"
    avcc = base.index(b"avcC") + 4
    yield "length_size_3", patch(base, avcc + 4, 0xFE, ">B"), 0, "lengthSizeMinusOne 2 is invalid"
    yield "avcc_sps_past_box", patch(base, avcc + 6, 0xFFFF, ">H"), 0, "avcC parameter set runs past its box"
    yield "no_avcc", rename(base, b"avcC", b"xvcC"), 0, "sample description 1 has no readable avcC box"
    yield "no_stsz", rename(base, b"stsz", b"xtsz"), 0, "lacks stsz, stsc or stco"
    yield "empty_stsd", patch(base, stsd + 12, 0), 0, "empty or truncated sample description"


@pytest.mark.parametrize("case", list(refusals()), ids=lambda c: c[0])
def test_damaged_or_unsupported_files_are_refused(case):
    from minivideo_b200 import front
    _, data, code, msg = case
    with pytest.raises(front.FrontError, match=msg) as e:
        front.Stream(data, "mp4")
    assert e.value.code == code, str(e.value)


# ---- a large file ------------------------------------------------------------------------------------------------

def _rss() -> int:
    with open("/proc/self/statm") as f:
        return int(f.read().split()[1]) * os.sysconf("SC_PAGE_SIZE")


def test_a_1000_picture_1080p_file_is_indexed_in_place():
    """About 1 GB of 1080p IDR pictures: the MP4 opens to the Annex-B stream's pictures and selection, and opening it
    does not copy the media data -- the NAL index points into the caller's buffer, so the process grows by far less
    than the file."""
    from helpers import split_nals
    from minivideo_b200 import front, synth
    s, _ = synth.generate(40, "1080p", want_soa=False, luma_cbp_percent=100, mean_coeffs_x10=220, level_scale_x10=30, seed=616)
    nals = split_nals(s)
    es = b"".join(nals[:2] + nals[2:] * 25) + bytes(4)
    del s, nals
    mp4 = mux(es + bytes(60), chunk_pattern=(7, 5), co64=True)
    assert len(mp4) > 900 << 20
    before = _rss()
    a = front.Stream(mp4, "mp4")
    grown = _rss() - before
    assert grown < 64 << 20, grown
    b = front.Stream(es)
    assert a.n_idr == b.n_idr == 1000
    for mode in (0, 1, 2):
        for n in (1, 9, 100, 1000):
            assert np.array_equal(a.select_idr(n, mode), b.select_idr(n, mode)), (n, mode)
    idx = np.array([0, 517, 999], np.int32)
    pa, pb = a.parse(indices=idx), b.parse(indices=idx)
    for f in FIELDS:
        assert np.array_equal(getattr(pa, f), getattr(pb, f)), f
