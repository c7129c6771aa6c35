"""MPEG-2 transport stream input of the host front end (mvf_open_ts): a TS whose video PID carries an Annex-B stream
opens to the same stream -- pictures, parameter generations, selection and parsed macroblocks -- as that stream, for
every variant tests/ts_mux.py writes; damage drops exactly the NAL units it touches; refusals carry a code and a
message; container detection (mvt_container) keeps every Annex-B input on its path."""
import ctypes as C
import os
import random
from pathlib import Path

import numpy as np
import pytest

from container_cases import FIELDS, NAMES, assert_same_stream, stream
from ts_mux import mux, surviving, with_aud_sei

ROOT = Path(__file__).resolve().parent.parent

KNOBS = {
    "plain": dict(),
    "m2ts_192": dict(packet_size=192),
    "parity_204": dict(packet_size=204),
    "psi_repeated": dict(psi_every=9),
    "psi_spanning": dict(psi_span=True, psi_every=25),
    "audio_first_program": dict(programs="audio_first"),
    "two_video_programs": dict(programs="two_video"),
    "audio_interleaved": dict(audio=True),
    "unbounded_pes": dict(bounded=False),
    "split_access_units": dict(pes_per_au=4),
    "split_unbounded": dict(pes_per_au=3, bounded=False),
    "stuffing": dict(stuffing=2),
    "null_packets": dict(null_packets=True),
    "duplicates": dict(dup=(0, 3, 7, 20)),
    "everything_192": dict(packet_size=192, psi_every=11, psi_span=True, audio=True, pes_per_au=2, stuffing=3,
                           null_packets=True, dup=(5,)),
}


@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("knob", sorted(KNOBS))
def test_ts_opens_to_the_annexb_stream(knob, name):
    es = stream(name)
    assert_same_stream(mux(es, **KNOBS[knob]), "ts", es, True)


@pytest.mark.parametrize("name", NAMES)
def test_aud_and_sei_nal_units(name):
    es = with_aud_sei(stream(name))
    assert_same_stream(mux(es, pes_per_au=2, packet_size=204), "ts", es, True)


def test_cif_baseline_and_generator_soa():
    from minivideo_b200 import front, synth
    es, soa = synth.generate(5, "cif", seed=612)
    got = front.Stream(mux(es, audio=True), "ts").parse()
    for f in FIELDS:
        assert np.array_equal(getattr(got, f), getattr(soa, f)), f


# ---- damage --------------------------------------------------------------------------------------------------------

def _damaged_case(es: bytes, kw: dict):
    """Open the damaged TS and the Annex-B stream without the NAL units the damage touches; both hold the same
    pictures, with the same generations and macroblocks."""
    from minivideo_b200 import front
    info = {}
    ts = mux(es, info=info, **kw)
    want = surviving(es, info["lost"])
    a, b = front.Stream(ts, "ts"), front.Stream(want)
    assert a.n_idr == b.n_idr < front.Stream(es).n_idr
    gens = b.picture_generations()
    assert np.array_equal(a.picture_generations(), gens)
    assert np.array_equal(a.select_idr(a.n_idr, 0), b.select_idr(b.n_idr, 0))
    for g in set(gens.tolist()) - {-1}:
        idx = np.flatnonzero(gens == g).astype(np.int32)
        pa, pb = a.parse(indices=idx, tolerant=True), b.parse(indices=idx, tolerant=True)
        for f in FIELDS + ("status",):
            assert np.array_equal(getattr(pa, f), getattr(pb, f)), (g, f)


@pytest.mark.parametrize("kind", ["drop", "tei", "cut"])
@pytest.mark.parametrize("name", ["high", "multi_size"])
def test_damage_drops_exactly_the_nal_units_it_touches(kind, name):
    es = stream(name)
    rng = random.Random(f"{kind}/{name}")
    n_video = len(mux(es)) // 188                       # more than the video packets: indices are clipped below
    for trial in range(4):
        picks = tuple(sorted({rng.randrange(3, n_video // 2) for _ in range(1 + trial % 2)}))
        kw = {kind: picks, "pes_per_au": 1 + trial % 3}
        try:
            _damaged_case(es, kw)
        except AssertionError as e:
            raise AssertionError(f"{kind} {picks} {kw}: {e}") from e


def test_a_lost_sps_loses_the_pictures_that_need_it():
    """Dropping the packet that holds the second SPS of the multi_size stream: the pictures after it use the first
    generation's parameters no more -- they name a PPS whose SPS is gone or changed -- exactly as in the Annex-B
    stream without that SPS."""
    es = stream("multi_size")
    from ts_mux import access_units
    sps2 = es.index(b"\x00\x00\x00\x01\x67", 10)
    _damaged_case(es, dict(drop=(_first_packet_of_pes(es, access_units(es).index(sps2)),)))


def _first_packet_of_pes(es: bytes, k: int) -> int:
    """Index among the video packets of the first packet of PES k (one PES per access unit, 14-byte PES headers)."""
    from ts_mux import access_units
    au = access_units(es) + [len(es)]
    return sum((au[i + 1] - au[i] + 14 + 183) // 184 for i in range(k))


# ---- refusals ------------------------------------------------------------------------------------------------------

def _strip_pid(ts: bytes, pid: int) -> bytes:
    return b"".join(ts[i:i + 188] for i in range(0, len(ts), 188) if ((ts[i + 1] & 0x1F) << 8 | ts[i + 2]) != pid)


def _clear_pusi(ts: bytes, pid: int) -> bytes:
    b = bytearray(ts)
    for i in range(0, len(b), 188):
        if ((b[i + 1] & 0x1F) << 8 | b[i + 2]) == pid:
            b[i + 1] &= ~0x40
    return bytes(b)


def refusals():
    es = stream("high")
    base = mux(es)
    yield "scrambled", mux(es, scrambled=True), -1, "scrambled"
    yield "hevc", mux(es, video_type=0x24), -1, "stream_type 0x24, not H.264"
    yield "mpeg2_video", mux(es, video_type=0x02), -1, "stream_type 0x02, not H.264"
    yield "no_video", mux(es, programs="audio_only"), -1, "no video stream"
    yield "no_sync", bytes(random.Random(5).randrange(256) for _ in range(5000)), 0, "no sync bytes"
    yield "annexb_bytes", es, 0, "no sync bytes"
    yield "no_pat", _strip_pid(base, 0), 0, "no program association table"
    yield "no_pmt", _strip_pid(base, 0x1000), 0, "no program map table \\(PMT\\) for program 1"
    yield "no_pes", _clear_pusi(base, 0x100), 0, "carries no PES packet"
    bad_crc = bytearray(base)
    bad_crc[4 + 1 + 10] ^= 1                            # inside the only PAT: its CRC no longer holds
    yield "pat_crc", bytes(bad_crc), 0, "no program association table"


@pytest.mark.parametrize("case", list(refusals()), ids=lambda c: c[0])
def test_damaged_or_unsupported_streams_are_refused(case):
    from minivideo_b200 import front
    _, data, code, msg = case
    with pytest.raises(front.FrontError, match=msg) as e:
        front.Stream(data, "ts")
    assert e.value.code == code, str(e.value)


def test_a_bad_psi_copy_is_ignored_until_a_good_one_comes():
    """The first PAT and PMT fail their CRC; the repetitions that follow are good."""
    es = stream("high")
    ts = bytearray(mux(es, psi_every=6))
    ts[4 + 1 + 10] ^= 1                                 # first PAT
    ts[188 + 4 + 1 + 14] ^= 1                           # first PMT
    assert_same_stream(bytes(ts), "ts", es, True)


def test_lost_sync_is_found_again():
    """Junk bytes between two packets: the packets after them are found at the period again, and only the NAL unit
    the junk interrupts is lost (the continuity counters show no gap, so nothing else)."""
    from minivideo_b200 import front
    es = stream("high")
    ts = mux(es)
    k = 40 * 188
    damaged = ts[:k] + bytes(range(1, 60)) + ts[k:]
    a, b = front.Stream(damaged, "ts"), front.Stream(es)
    assert b.n_idr - 1 <= a.n_idr <= b.n_idr


# ---- a large stream ------------------------------------------------------------------------------------------------

def _rss() -> int:
    with open("/proc/self/statm") as f:
        return int(f.read().split()[1]) * os.sysconf("SC_PAGE_SIZE")


def test_a_1gb_ts_keeps_only_its_idr_bytes():
    """About 1 GB of 1080p: one IDR picture in 20, large non-IDR slices (type 1) between them.  The stream keeps a
    copy of the SPS, PPS and IDR NAL units only, so the process grows by about the IDR bytes, not the file size."""
    from helpers import split_nals
    from minivideo_b200 import front, synth
    s, _ = synth.generate(5, "1080p", want_soa=False, luma_cbp_percent=100, mean_coeffs_x10=220, level_scale_x10=30, seed=617)
    nals = split_nals(s)
    ps, idrs = nals[:2], nals[2:]
    rng = random.Random(7)
    filler = b"\x00\x00\x00\x01\x41" + bytes(rng.randrange(1, 256) for _ in range(1 << 20))
    parts = list(ps)
    idr_bytes = 0
    for k in range(50):
        parts.append(idrs[k % len(idrs)])
        idr_bytes += len(idrs[k % len(idrs)])
        parts += [filler] * 19
    es = b"".join(parts) + bytes(4)
    del s, nals, parts
    ts = mux(es, bounded=False)
    assert len(ts) > 900 << 20
    before = _rss()
    a = front.Stream(ts, "ts")
    grown = _rss() - before
    assert grown < idr_bytes + (48 << 20), (grown, idr_bytes)
    b = front.Stream(es)
    assert a.n_idr == b.n_idr == 50
    for mode in (0, 1, 2):
        for n in (1, 9, 50):
            assert np.array_equal(a.select_idr(n, mode), b.select_idr(n, mode)), (n, mode)
    idx = np.array([0, 27, 49], np.int32)
    pa, pb = a.parse(indices=idx), b.parse(indices=idx)
    for f in FIELDS:
        assert np.array_equal(getattr(pa, f), getattr(pb, f)), f


# ---- container detection -------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def shim():
    from minivideo_b200 import build
    build.build_thumbnailer()
    lib = C.CDLL(str(ROOT / "minivideo_b200" / "libminivideo_b200.so"))
    lib.mvt_container.argtypes = [C.c_char_p, C.c_size_t]
    return lib


ANNEXB, MP4, TS, MKV = 0, 1, 2, 3


def detection_cases():
    from mkv_mux import mux as mkv
    from mp4_mux import mux as mp4
    es = stream("high")
    ts = mux(es)
    yield "annexb", es, ANNEXB
    yield "annexb_3byte", es[1:], ANNEXB
    yield "mp4", mp4(es), MP4
    yield "mkv", mkv(es), MKV
    yield "ts_188", ts, TS
    yield "m2ts_192", mux(es, packet_size=192), TS
    yield "ts_204", mux(es, packet_size=204), TS
    yield "ts_cut_mid_packet", ts[100:], TS
    yield "ts_four_packets", ts[:4 * 188], ANNEXB
    yield "start_code_then_sync_period", b"\x00\x00\x01\x09" + ts[4:], ANNEXB
    yield "start_code4_then_sync_period", b"\x00\x00\x00\x01" + ts[4:], ANNEXB
    yield "ebml_magic_only", b"\x1a\x45\xdf\xa3", MKV
    yield "random", bytes(random.Random(3).randrange(256) for _ in range(4000)), ANNEXB
    yield "empty", b"", ANNEXB


@pytest.mark.parametrize("case", list(detection_cases()), ids=lambda c: c[0])
def test_container_detection(shim, case):
    _, data, want = case
    assert shim.mvt_container(data, len(data)) == want


def test_every_annexb_golden_stream_stays_annexb(shim):
    from helpers import paramset_change_stream
    from minivideo_b200 import synth
    n = 0
    for path in sorted((ROOT / "tests" / "golden").glob("*.npz")):
        z = np.load(path, allow_pickle=False)
        if "stream" not in z.files:
            continue
        data = z["stream"].tobytes()
        assert shim.mvt_container(data, len(data)) == ANNEXB, path.name
        n += 1
    assert n >= 10
    for data in (paramset_change_stream(True)[0], synth.generate(3, "cif", seed=9)[0]):
        assert shim.mvt_container(data, len(data)) == ANNEXB


@pytest.mark.parametrize("name,data_kind,ok", [
    ("x.ts", "ts", True), ("x.M2TS", "ts", True), ("x.mts", "ts", True), ("x.m2t", "ts", True),
    ("x.mkv", "mkv", True), ("x.MK3D", "mkv", True), ("x.webm", "mkv", True),
    ("x.ts", "annexb", False), ("x.mkv", "mp4", False), ("x.webm", "ts", False), ("x.m2ts", "mkv", False),
    ("x.avi", "ts", False),
])
def test_drop_in_parse_accepts_a_container_name_only_with_its_content(shim, tmp_path, name, data_kind, ok):
    from mkv_mux import mux as mkv
    from mp4_mux import mux as mp4
    es = stream("high")
    data = {"ts": lambda: mux(es), "mkv": lambda: mkv(es), "mp4": lambda: mp4(es), "annexb": lambda: es}[data_kind]()
    (tmp_path / name).write_bytes(data)
    media = C.c_void_p()
    assert shim.minivideo_open(str(tmp_path / name).encode(), C.byref(media)) == 1
    assert shim.minivideo_parse(media, False, True, False) == int(ok)
    assert shim.minivideo_close(C.byref(media)) == 1
