"""MP4 input end to end on the GPU: mv_thumbnailer and the drop-in library write, byte for byte, the same picture files
for an MP4 file as for the Annex-B stream that holds the same NAL units (the MP4 goes through mvf_open_mp4, the rest
of the path -- selection, CAVLC, packed transfer, kf_recon, file writers -- is the one the Annex-B tests pin)."""
import ctypes as C
import os
import subprocess
import tempfile
from pathlib import Path

import pytest

from mp4_mux import es_twin, mux, nal_units
from oracle import ref

ROOT = Path(__file__).resolve().parent.parent
MV = ROOT / "minivideo_b200" / "mv_thumbnailer"


@pytest.fixture(scope="module")
def cli():
    from minivideo_b200 import build
    return build.build_thumbnailer()


def _tmp():
    return tempfile.TemporaryDirectory(dir="/dev/shm" if os.path.isdir("/dev/shm") else None)


def _run(exe, name: str, data: bytes, args: list[str], out_flag: bool = True):
    """Run one CLI in a scratch directory on `data` stored as `name`; ({file name: bytes}, finished process)."""
    with _tmp() as d:
        (Path(d) / name).write_bytes(data)
        r = subprocess.run([str(exe), "-i", str(Path(d) / name)] + args + (["-o", d] if out_flag else []),
                           capture_output=True, text=True, cwd=d)
        return {p.name: p.read_bytes() for p in Path(d).iterdir() if p.name != name and not p.name.startswith("core")}, r


MODES = ("unfiltered", "ordered", "distributed")


def _same_files(es: bytes, mp4: bytes, args: list[str], n: int, mode: str = "unfiltered"):
    """mv_thumbnailer -n n -e mode on both forms: the same files, one per picture the selection picks (the reference's
    'distributed' steps through the candidates by an integer quotient and can pick fewer than n, filter.c:140)."""
    from minivideo_b200 import front
    args = args + ["-n", str(n), "-e", mode]
    want, r1 = _run(MV, "in.264", es, args)
    got, r2 = _run(MV, "in.mp4", mp4, args)
    assert r1.returncode == 0 and r2.returncode == 0, (r1.stderr[-1500:], r2.stderr[-1500:])
    n_files = len(front.Stream(es).select_idr(n, MODES.index(mode)))
    assert n_files >= 1
    assert sorted(got) == sorted(want) and len(want) == n_files, (sorted(want), sorted(got), n_files)
    for name in want:
        assert got[name] == want[name], name


def _cif():
    from minivideo_b200 import synth
    return synth.generate(12, "cif", seed=901)[0]


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["jpg", "png", "bmp", "tga", "yuv420", "yuv444"])
@pytest.mark.parametrize("mode", MODES)
def test_cli_writes_the_same_files_for_mp4_and_annexb(cli, fmt, mode):
    es = _cif()
    _same_files(es_twin(es), mux(es, chunk_pattern=(2, 3), co64=True), ["-f", fmt], 4, mode)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["bmp", "png"])
def test_cli_scaled_thumbnails_from_mp4(cli, fmt):
    es = _cif()
    _same_files(es_twin(es), mux(es, moov_first=False), ["-f", fmt, "-s", "4"], 3)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["yuv420", "bmp"])
def test_cli_follows_sample_descriptions(cli, fmt):
    """Two avc1 sample descriptions with other scaling lists, chroma QP offsets and picture size, selected through
    stsc: each picture comes out with its own description's parameters and size, as from the Annex-B stream."""
    from minivideo_b200 import synth
    a = synth.generate(3, width_mbs=6, height_mbs=4, profile_idc=100, transform8x8=1, scaling_lists=1,
                       cb_qp_offset=4, cr_qp_offset=-6, seed=613)[0]
    b = synth.generate(4, width_mbs=9, height_mbs=5, profile_idc=100, transform8x8=0, scaling_lists=1,
                       cb_qp_offset=-2, cr_qp_offset=5, seed=614)[0]
    es = a.rstrip(b"\x00") + b
    mp4 = mux(es, chunk_pattern=(2,), audio_first=True)
    assert mp4.count(b"avc1") == 3          # the ftyp brand and two sample descriptions
    for extra in ([], ["-b", "2"]):
        _same_files(es_twin(es), mp4, ["-f", fmt] + extra, 7)


@pytest.mark.gpu
def test_cli_three_generations_and_junk_non_sync_samples(cli):
    """The multi_paramsets stream with random type-1 NAL units in non-sync samples between the IDR samples, AUD and
    SEI NAL units inside them, and one sample whose length field runs past its end."""
    from helpers import paramset_change_stream
    from minivideo_b200 import synth
    es = paramset_change_stream(True)[0]
    other = nal_units(synth.generate(1, width_mbs=7, height_mbs=3, profile_idc=66, seed=615)[0])
    for kw in (dict(junk_samples=2), dict(junk_samples=1, damaged_sample=(4, [other[0], other[2]])),
               dict(aud_sei=True, length_size=2)):
        mp4 = mux(es, chunk_pattern=(3, 1), **kw)
        _same_files(es_twin(es), mp4, ["-f", "bmp"], 6)
        if "aud_sei" not in kw:
            _same_files(es_twin(es), mp4, ["-f", "yuv420"], 3, "ordered")


@pytest.mark.gpu
def test_drop_in_library_decodes_mp4_like_annexb(cli):
    """minivideo_open / parse / decode through ctypes on x.mp4 write the files they write on x.264."""
    lib = C.CDLL(str(ROOT / "minivideo_b200" / "libminivideo_b200.so"))
    es = _cif()
    mp4 = mux(es, chunk_pattern=(4,))
    outs = []
    for name, data in (("x.264", es_twin(es)), ("x.mp4", mp4), ("x.MOV", mp4)):
        with _tmp() as d:
            (Path(d) / name).write_bytes(data)
            media = C.c_void_p()
            assert lib.minivideo_open(str(Path(d) / name).encode(), C.byref(media)) == 1
            assert lib.minivideo_parse(media, False, True, False) == 1, name
            assert lib.minivideo_decode(media, d.encode(), 1, 75, 5, 1) == 1, name        # PICTURE_BMP, 5, ordered
            assert lib.minivideo_close(C.byref(media)) == 1
            outs.append({p.name: p.read_bytes() for p in Path(d).iterdir() if p.name != name})
    assert len(outs[0]) == 5 and outs[0] == outs[1] == outs[2]


@pytest.mark.gpu
def test_reference_cli_on_the_same_mp4(cli):
    """Where oracle/_ref is built: the reference's own mini_thumbnailer, through its own MP4 demuxer, against
    mv_thumbnailer on the same MP4 file."""
    if not ref.MINI_THUMBNAILER.exists():
        pytest.skip("reference CLI build is not present")
    es = _cif()
    mp4 = mux(es)
    args = ["-f", "yuv420", "-n", "4", "-e", "unfiltered"]
    want, r1 = _run(ref.MINI_THUMBNAILER, "in.mp4", mp4, args, out_flag=False)
    got, r2 = _run(MV, "in.mp4", mp4, args)
    assert r1.returncode == 0 and r2.returncode == 0, (r1.stdout[-1500:], r1.stderr[-1500:], r2.stderr[-1500:])
    assert sorted(want) == sorted(got)
    for name in want:
        assert want[name] == got[name], name
