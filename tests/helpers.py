"""Shared helpers for the tests."""
from __future__ import annotations

import functools
import hashlib
import json
import os
import struct
import zlib
from pathlib import Path

import numpy as np

GOLDEN = Path(__file__).resolve().parent / "golden"


def golden_names():
    """Single-generation fixtures (one SPS/PPS pair); multi_*.npz hold streams whose parameter sets change."""
    return sorted(p.stem for p in GOLDEN.glob("*.npz") if not p.stem.startswith("multi_"))


def load_golden(name):
    """Returns (Soa built from the REFERENCE's parse, fixture dict)."""
    from minivideo_b200.synth import Soa
    z = np.load(GOLDEN / f"{name}.npz")
    soa = Soa(int(z["width_mbs"]), int(z["height_mbs"]), int(z["n_pics"]), z["soa_mb_kind"], z["soa_i16_mode"],
              z["soa_chroma_mode"], z["soa_qp_y"], z["soa_cbp"], z["soa_luma_modes"], z["soa_coeff"],
              cb_qp_offset=int(z["cb_qp_offset"]), cr_qp_offset=int(z["cr_qp_offset"]))
    return soa, z


def large_digests():
    return json.loads((GOLDEN / "large_digests.json").read_text())


def sha(a) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def digest(b: bytes) -> str:
    return hashlib.sha256(b).hexdigest()


# Expected results of the tests that compare with the reference's binaries, for machines without oracle/_ref.  Where
# they come from: the reference's sources were not available when the file was made, so it was recorded with
# MVG_RECORD_REFERENCE from this project's own writers, mv_thumbnailer, front end and CPU oracle standing in for the
# reference binaries, at the code whose GPU suite last passed against the built reference.  Until it is re-recorded
# from the reference itself it therefore pins this project's results; every run where oracle/_ref is built checks
# each stored entry against the reference and fails on a difference.
REFERENCE_OUTPUTS = GOLDEN / "reference_outputs.json"


def reference_output(key: str, live, available: bool):
    """The result for one test case of the reference's binaries (oracle/_ref, built by oracle/Makefile from the
    reference's sources, which are not part of this repository), as JSON data: SHA-256 digests of files and arrays,
    picture indices.  Where they are built, live() runs them and the result must equal the entry stored in
    golden/reference_outputs.json; elsewhere the stored entry stands in (see REFERENCE_OUTPUTS for its source).  With
    MVG_RECORD_REFERENCE=FILE every live result is collected into FILE instead of being checked: run the suite so
    where oracle/_ref is built, and copy FILE over golden/reference_outputs.json to re-record it."""
    recorded = _recorded_reference_outputs()
    if available:
        out = live()
        rec_path = os.environ.get("MVG_RECORD_REFERENCE")
        if rec_path:
            rec = json.loads(Path(rec_path).read_text()) if Path(rec_path).exists() else {}
            rec[key] = out
            Path(rec_path).write_text(json.dumps(rec, indent=1, sort_keys=True) + "\n")
        else:
            assert key in recorded and recorded[key] == out, f"golden/reference_outputs.json differs from the reference for {key!r}"
        return out
    assert key in recorded, f"no stored reference output for {key!r} (tests/golden/reference_outputs.json)"
    return recorded[key]


@functools.lru_cache(maxsize=None)
def _recorded_reference_outputs() -> dict:
    return json.loads(REFERENCE_OUTPUTS.read_text())


def oracle_sps_from_tables(soa, ls4, ls8):
    import ctypes as C
    from oracle import cpu
    s = cpu.OracleSps()
    s.width_mbs, s.height_mbs = soa.width_mbs, soa.height_mbs
    a = np.ascontiguousarray(ls4, np.int32); b = np.ascontiguousarray(ls8, np.int32)
    C.memmove(s.ls4, a.ctypes.data, a.nbytes)
    C.memmove(s.ls8, b.ctypes.data, b.nbytes)
    s.cb_qp_offset, s.cr_qp_offset = soa.cb_qp_offset, soa.cr_qp_offset
    return s


def oracle_reconstruct_with_tables(soa, ls4, ls8, want_residual=False):
    """Oracle reconstruction using explicit LevelScale tables (e.g. the reference's own)."""
    import ctypes as C
    from oracle import cpu
    L = cpu.lib()
    sps = oracle_sps_from_tables(soa, ls4, ls8)
    W, H, N = soa.width, soa.height, soa.n_mbs
    yuv = np.zeros((soa.n_pics, W * H * 3 // 2), np.uint8)
    res = np.zeros((soa.n_pics * N, 384), np.int16) if want_residual else None
    p_ = lambda a: a.ctypes.data_as(C.c_void_p)
    for p in range(soa.n_pics):
        s = slice(p * N, (p + 1) * N)
        arrs = [np.ascontiguousarray(x[s]) for x in (soa.mb_kind, soa.i16_mode, soa.chroma_mode, soa.qp_y, soa.luma_modes, soa.coeff)]
        y = yuv[p, :W * H]; cb = yuv[p, W * H:W * H * 5 // 4]; cr = yuv[p, W * H * 5 // 4:]
        r = res[s] if want_residual else None
        L.oracle_reconstruct_picture(C.byref(sps), *[p_(a) for a in arrs], p_(y), p_(cb), p_(cr),
                                     p_(r) if r is not None else None)
    return yuv, res


def png_decode(png: bytes) -> np.ndarray:
    """Minimal PNG reader (8-bit truecolour, no interlace) -- independent of both writers."""
    assert png[:8] == bytes([137, 80, 78, 71, 13, 10, 26, 10])
    pos, idat, w, h = 8, b"", 0, 0
    while pos < len(png):
        n, tag = struct.unpack(">I4s", png[pos:pos + 8])
        body = png[pos + 8:pos + 8 + n]
        assert struct.unpack(">I", png[pos + 8 + n:pos + 12 + n])[0] == zlib.crc32(tag + body)
        if tag == b"IHDR":
            w, h, depth, ctype, comp, filt, lace = struct.unpack(">IIBBBBB", body)
            assert (depth, ctype, comp, filt, lace) == (8, 2, 0, 0, 0)
        elif tag == b"IDAT":
            idat += body
        pos += 12 + n
    raw = np.frombuffer(zlib.decompress(idat), np.uint8).reshape(h, 3 * w + 1)
    out = np.zeros((h, 3 * w), np.int32)
    for y in range(h):
        f, line = int(raw[y, 0]), raw[y, 1:].astype(np.int32)
        up = out[y - 1] if y else np.zeros(3 * w, np.int32)
        if f == 0:
            out[y] = line
        elif f == 2:
            out[y] = (line + up) & 255
        else:
            for i in range(3 * w):
                a = out[y, i - 3] if i >= 3 else 0
                c = up[i - 3] if i >= 3 else 0
                b = up[i]
                if f == 1:
                    pred = a
                elif f == 3:
                    pred = (a + b) >> 1
                else:
                    p = a + b - c
                    pa, pb, pc = abs(p - a), abs(p - b), abs(p - c)
                    pred = a if pa <= pb and pa <= pc else (b if pb <= pc else c)
                out[y, i] = (line[i] + pred) & 255
    return out.reshape(h, w, 3).astype(np.uint8)


def split_nals(stream: bytes) -> list[bytes]:
    """NAL units of a generated stream (4-byte start codes, 64 bytes of zero padding at the end), start codes included."""
    body = stream.rstrip(b"\x00")
    # a NAL may end in zero bytes that rstrip took: the generator never ends one that way (rbsp_trailing_bits)
    parts = body.split(b"\x00\x00\x00\x01")[1:]
    return [b"\x00\x00\x00\x01" + p for p in parts]


PAD = b"\x00" * 64


def paramset_change_stream(geometry_change: bool = False):
    """A stream whose parameter sets change between IDR pictures, the way BASELINE.md's chunk files do when their
    headers differ: segment A (SPS + PPS + 2 pictures), segment B (a new SPS with other scaling lists and a new PPS with
    other chroma QP offsets and pic_init_qp, 2 pictures), segment C (only a new PPS, 2 pictures).  With
    geometry_change the second SPS also changes the picture size.  Returns (stream, [per-segment Soa])."""
    from minivideo_b200 import synth
    geo_a = dict(width_mbs=6, height_mbs=4)
    geo_b = dict(width_mbs=8, height_mbs=5) if geometry_change else geo_a
    common = dict(profile_idc=100, transform8x8=1, scaling_lists=1, qp_min=12, qp_max=44)
    a, soa_a = synth.generate(2, seed=301, init_qp=26, cb_qp_offset=0, cr_qp_offset=0, **geo_a, **common)
    b, soa_b = synth.generate(2, seed=302, init_qp=33, cb_qp_offset=5, cr_qp_offset=-4, **geo_b, **common)
    c, soa_c = synth.generate(2, seed=302, init_qp=21, cb_qp_offset=-3, cr_qp_offset=2, **geo_b, **common)
    nb, nc = split_nals(b), split_nals(c)
    assert nb[0][4] == 0x67 and nc[0] == nb[0], "segments B and C must carry the same SPS"
    stream = b"".join(split_nals(a)) + b"".join(nb) + b"".join(nc[1:]) + PAD
    return stream, [soa_a, soa_b, soa_c]
