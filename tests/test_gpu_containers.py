"""Transport stream and Matroska input end to end on the GPU: mv_thumbnailer and the drop-in library write, byte for
byte, the same picture files for a 188-byte TS, a 192-byte M2TS and a Matroska file as for the Annex-B stream that
holds the same NAL units (the container goes through mvf_open_ts / mvf_open_mkv, the rest of the path -- selection,
CAVLC, packed transfer, kf_recon, file writers -- is the one the Annex-B tests pin)."""
import ctypes as C
import os
import subprocess
import tempfile
from pathlib import Path

import pytest

import mkv_mux
import ts_mux
from oracle import ref

ROOT = Path(__file__).resolve().parent.parent
MV = ROOT / "minivideo_b200" / "mv_thumbnailer"
MODES = ("unfiltered", "ordered", "distributed")


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


def _forms(es: bytes):
    """(file name, bytes, Annex-B twin) of the three container forms of `es`."""
    return [("in.ts", ts_mux.mux(es, audio=True, psi_every=40), es),
            ("in.m2ts", ts_mux.mux(es, packet_size=192, pes_per_au=2, bounded=False), es),
            ("in.mkv", mkv_mux.mux(es, lacing="xiph", per_block=2, cluster_unknown=True), mkv_mux.es_twin(es))]


def _same_files(es: bytes, name: str, data: bytes, args: list[str], n: int, mode: str = "unfiltered"):
    """mv_thumbnailer -n n -e mode on both forms: the same files, one per picture the front end's selection picks."""
    from minivideo_b200 import front
    args = args + ["-n", str(n), "-e", mode]
    want, r1 = _run(MV, "in.264", es, args)
    got, r2 = _run(MV, name, data, args)
    assert r1.returncode == 0 and r2.returncode == 0, (r1.stderr[-1500:], r2.stderr[-1500:])
    n_files = len(front.Stream(es).select_idr(n, MODES.index(mode)))
    assert n_files >= 1
    assert sorted(got) == sorted(want) and len(want) == n_files, (sorted(want), sorted(got), n_files)
    for f in want:
        assert got[f] == want[f], f


def _cif():
    from minivideo_b200 import synth
    return synth.generate(12, "cif", seed=901)[0]


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["png", "yuv420"])
@pytest.mark.parametrize("mode", MODES)
def test_cli_writes_the_same_files_for_ts_m2ts_mkv_and_annexb(cli, fmt, mode):
    for name, data, twin in _forms(_cif()):
        _same_files(twin, name, data, ["-f", fmt], 4, mode)


@pytest.mark.gpu
def test_cli_scaled_thumbnails(cli):
    for name, data, twin in _forms(_cif()):
        _same_files(twin, name, data, ["-f", "bmp", "-s", "4"], 3)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["yuv420", "png"])
def test_cli_follows_parameter_generations_that_change_the_picture_size(cli, fmt):
    """The multi_size stream: the second SPS changes the picture size between pictures."""
    from helpers import paramset_change_stream
    es = paramset_change_stream(True)[0]
    for name, data, twin in _forms(es):
        _same_files(twin, name, data, ["-f", fmt], 6)
        _same_files(twin, name, data, ["-f", fmt, "-b", "2"], 3, "ordered")


@pytest.mark.gpu
def test_drop_in_library_decodes_ts_and_mkv_like_annexb(cli):
    """minivideo_open / parse / decode through ctypes on x.ts, x.m2ts, x.MKV and x.webm write the files they write on
    the Annex-B twin."""
    lib = C.CDLL(str(ROOT / "minivideo_b200" / "libminivideo_b200.so"))
    es = _cif()
    ts, m2ts, mkv = (f[1] for f in _forms(es))
    for twin, cases in ((es, [("x.ts", ts), ("x.m2ts", m2ts)]), (mkv_mux.es_twin(es), [("x.MKV", mkv), ("x.webm", mkv)])):
        outs = []
        for name, data in [("x.264", twin)] + cases:
            with _tmp() as d:
                (Path(d) / name).write_bytes(data)
                media = C.c_void_p()
                assert lib.minivideo_open(str(Path(d) / name).encode(), C.byref(media)) == 1
                assert lib.minivideo_parse(media, False, True, False) == 1, name
                assert lib.minivideo_decode(media, d.encode(), 3, 75, 5, 2) == 1, name        # PICTURE_PNG, 5, distributed
                assert lib.minivideo_close(C.byref(media)) == 1
                outs.append({p.name: p.read_bytes() for p in Path(d).iterdir() if p.name != name})
        from minivideo_b200 import front
        assert len(outs[0]) == len(front.Stream(twin).select_idr(5, 2)) >= 1
        assert all(o == outs[0] for o in outs[1:])


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["ts", "mkv"])
def test_reference_cli_on_the_same_file(cli, kind):
    """Where oracle/_ref is built: the reference's own mini_thumbnailer, through its own demuxer, against
    mv_thumbnailer on the same file."""
    if not ref.MINI_THUMBNAILER.exists():
        pytest.skip("reference CLI build is not present")
    es = _cif()
    name, data = ("in.ts", ts_mux.mux(es)) if kind == "ts" else ("in.mkv", mkv_mux.mux(es))
    args = ["-f", "yuv420", "-n", "4", "-e", "unfiltered"]
    want, r1 = _run(ref.MINI_THUMBNAILER, name, data, args, out_flag=False)
    got, r2 = _run(MV, name, data, args)
    assert r1.returncode == 0 and r2.returncode == 0, (r1.stdout[-1500:], r1.stderr[-1500:], r2.stderr[-1500:])
    assert sorted(want) == sorted(got)
    for f in want:
        assert want[f] == got[f], f
