"""mv_thumbnailer (bitstream -> front end -> C ABI -> picture files) against the files the unmodified
reference CLI (oracle/_ref/mini_thumbnailer) writes for the same stream and arguments: byte for byte (SHA-256), live
where oracle/_ref is built, elsewhere against the digests stored in tests/golden/reference_outputs.json (where they
come from: tests/helpers.py, REFERENCE_OUTPUTS)."""
import os
import subprocess
import tempfile
from pathlib import Path

import numpy as np
import pytest

from helpers import digest, reference_output
from oracle import ref

ROOT = Path(__file__).resolve().parent.parent
MV = ROOT / "minivideo_b200" / "mv_thumbnailer"


@pytest.fixture(scope="module")
def cli():
    from minivideo_b200 import build
    return build.build_thumbnailer()


def test_cli_builds_and_rejects_bad_arguments(cli):
    assert os.access(cli, os.X_OK)
    assert subprocess.run([str(cli)], capture_output=True).returncode == 2
    assert subprocess.run([str(cli), "-i", "x.264", "-f", "webp"], capture_output=True).returncode == 2
    r = subprocess.run([str(cli), "-i", "/nonexistent.264"], capture_output=True, text=True)
    assert r.returncode == 1 and "cannot open" in r.stderr


SHIM_CLI = ROOT / "oracle" / "_ref" / "mini_thumbnailer_b200"     # the reference's main.cpp linked against our library


def test_drop_in_library_exports_the_reference_entry_points(cli):
    """libminivideo_b200.so: every function of minivideo/src/minivideo.h:89-149, callable without a GPU
    up to the point where decoding starts."""
    import ctypes as C
    lib = C.CDLL(str(ROOT / "minivideo_b200" / "libminivideo_b200.so"))
    for name in ("minivideo_print_infos", "minivideo_get_infos", "minivideo_endianness", "minivideo_open",
                 "minivideo_parse", "minivideo_decode", "minivideo_extract", "minivideo_close"):
        assert hasattr(lib, name), name
    assert lib.minivideo_endianness() == 1234
    media = C.c_void_p()
    assert lib.minivideo_open(b"/nonexistent.264", C.byref(media)) == 0 and not media
    from minivideo_b200 import synth
    stream, _ = synth.generate(1, "cif", seed=3)
    with tempfile.TemporaryDirectory() as d:
        for name, parse_ok in (("a.264", 1), ("a.mp4", 0)):
            (Path(d) / name).write_bytes(stream)
            assert lib.minivideo_open(str(Path(d) / name).encode(), C.byref(media)) == 1
            assert lib.minivideo_parse(media, False, True, False) == parse_ok
            if parse_ok:
                assert lib.minivideo_decode(media, b"", 4, 75, 1, 0) == 0        # PICTURE_WEBP: not supported
            assert lib.minivideo_close(C.byref(media)) == 1 and not media


@pytest.mark.gpu
@pytest.mark.parametrize("fmt,n,mode", [("yuv420", 1, "unfiltered"), ("bmp", 3, "unfiltered"), ("tga", 4, "ordered"),
                                        ("png", 2, "unfiltered"), ("jpg", 2, "unfiltered"), ("yuv444", 2, "ordered")])
def test_reference_cli_linked_against_the_drop_in_library(cli, fmt, n, mode):
    """The reference's own mini_thumbnailer main.cpp, unmodified, linked against libminivideo_b200.so, writes
    the files the reference build of the same program writes."""
    from minivideo_b200 import synth
    if not (SHIM_CLI.exists() and ref.MINI_THUMBNAILER.exists()):
        pytest.skip("reference CLI builds are not present")
    stream, _ = synth.generate(9, "cif", seed=905)
    args = ["-f", fmt, "-n", str(n), "-e", mode]
    (want, r1), (got, r2) = _run(ref.MINI_THUMBNAILER, stream, args), _run(SHIM_CLI, stream, args)
    assert r1.returncode == 0 and r2.returncode == 0, (r1.stderr[-1500:], r2.stderr[-1500:])
    assert sorted(want) == sorted(got) and len(want) == n
    for name in want:
        assert want[name] == got[name], name


def _run(exe, stream: bytes, args: list[str]):
    """Run one CLI in a scratch directory on the stream; return ({file name: bytes}, the finished process)."""
    with tempfile.TemporaryDirectory(dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as d:
        (Path(d) / "in.264").write_bytes(stream)
        r = subprocess.run([str(exe), "-i", str(Path(d) / "in.264")] + args, capture_output=True, text=True, cwd=d)
        return {p.name: p.read_bytes() for p in Path(d).iterdir() if p.name != "in.264"}, r


def _reference_files(stream: bytes, args: list[str], may_crash: bool = False, keep=lambda data: True):
    """{file name: SHA-256} of the files the reference CLI writes, core dumps left out; a file `keep` rejects maps to None."""
    def live():
        files, r = _run(ref.MINI_THUMBNAILER, stream, args)
        assert may_crash or r.returncode == 0, (r.stdout[-1500:], r.stderr[-1500:])
        return {k: digest(v) if keep(v) else None for k, v in files.items() if not k.startswith("core")}
    return reference_output(f"mini_thumbnailer {digest(stream)[:16]} {' '.join(args)}", live, ref.MINI_THUMBNAILER.exists())


def _run_both(stream: bytes, args: list[str], ref_may_crash: bool = False):
    """The files the reference CLI and mv_thumbnailer write for the same stream and arguments, {file name: SHA-256} each."""
    files, r = _run(MV, stream, args + ["-o", "."])
    assert r.returncode == 0, (r.stdout[-1500:], r.stderr[-1500:])
    return _reference_files(stream, args, ref_may_crash), {k: digest(v) for k, v in files.items()}


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["yuv420", "bmp", "tga", "png", "yuv444"])
@pytest.mark.parametrize("mode,n", [("unfiltered", 1), ("unfiltered", 5), ("ordered", 4), ("distributed", 4)])
def test_cli_files_equal_the_reference_cli(cli, fmt, mode, n):
    from minivideo_b200 import synth
    stream, _ = synth.generate(12, "cif", seed=901)
    # 'distributed' indexes one past its candidate list in the reference (demuxer/filter.c:179-186) and
    # can abort after writing some of the pictures: compare what it did write
    crashy = mode == "distributed"
    want, got = _run_both(stream, ["-f", fmt, "-n", str(n), "-e", mode], ref_may_crash=crashy)
    if crashy:
        assert set(want) <= set(got) and len(want) >= n - 1
        want.pop(sorted(want)[-1])          # the last file may be cut short by the abort
    else:
        assert sorted(want) == sorted(got)
    for name in want:
        assert want[name] == got[name], name


@pytest.mark.gpu
@pytest.mark.parametrize("args", [[], ["-f", "jpg"]], ids=["default", "jpg"])
def test_cli_default_format_and_jpg_are_written_as_png_like_the_reference_build(cli, args):
    """mini_thumbnailer defaults to 'jpg' (main.cpp:56); the reference build without libjpeg writes PNG files for
    it (export.c:652-657) through its vendored stb writer."""
    from minivideo_b200 import synth
    stream, _ = synth.generate(3, width_mbs=20, height_mbs=12, profile_idc=100, transform8x8=1, scaling_lists=1, seed=911)
    want, got = _run_both(stream, args + ["-n", "3"])
    assert sorted(want) == sorted(got) == ["in_0.png", "in_1.png", "in_2.png"]
    assert want == got


@pytest.mark.gpu
def test_cli_high_profile_stream_and_small_batches(cli):
    from minivideo_b200 import synth
    stream, _ = synth.generate(7, width_mbs=20, height_mbs=12, profile_idc=100, transform8x8=1, scaling_lists=1,
                               cb_qp_offset=3, cr_qp_offset=-1, seed=902)
    want, _ = _run_both(stream, ["-f", "bmp", "-n", "7"])
    for batch in ("1", "3", "64"):
        _, got = _run_both(stream, ["-f", "bmp", "-n", "7", "-b", batch])
        assert want == got, batch


@pytest.mark.gpu
def test_cli_scaled_thumbnail_is_the_box_average(cli):
    """-s has no reference counterpart: defined as the rounded box average of the scale-1 RGB picture."""
    from minivideo_b200 import synth
    stream, _ = synth.generate(1, "cif", seed=903)
    with tempfile.TemporaryDirectory() as d:
        (Path(d) / "in.264").write_bytes(stream)
        for s in (1, 4):
            r = subprocess.run([str(MV), "-i", str(Path(d) / "in.264"), "-f", "bmp", "-s", str(s), "-o", d], capture_output=True, text=True)
            assert r.returncode == 0, r.stderr
            os.rename(Path(d) / "in.bmp", Path(d) / f"s{s}.bmp")

        def bmp(p):
            raw = np.fromfile(p, np.uint8)
            w, h = int(raw[18:22].view("<u4")[0]), int(raw[22:26].view("<u4")[0])
            return raw[54:].reshape(h, w * 3)[::-1].reshape(h, w, 3).astype(np.uint32)
        full, small = bmp(Path(d) / "s1.bmp"), bmp(Path(d) / "s4.bmp")
        h, w = full.shape[:2]
        assert np.array_equal(small, (full.reshape(h // 4, 4, w // 4, 4, 3).sum(axis=(1, 3)) + 8) // 16)


@pytest.mark.gpu
def test_cli_scaled_png_and_unwritable_directory(cli):
    """-s with PNG output holds the same pixels as -s with BMP output; an unwritable output directory is an error
    exit, not a silent success."""
    from minivideo_b200 import synth
    stream, _ = synth.generate(2, "cif", seed=913)
    with tempfile.TemporaryDirectory() as d:
        (Path(d) / "in.264").write_bytes(stream)
        for fmt in ("png", "bmp"):
            r = subprocess.run([str(MV), "-i", str(Path(d) / "in.264"), "-f", fmt, "-n", "2", "-s", "2", "-o", d], capture_output=True, text=True)
            assert r.returncode == 0, r.stderr
        from helpers import png_decode
        png = png_decode((Path(d) / "in_1.png").read_bytes())
        bmp = np.fromfile(Path(d) / "in_1.bmp", np.uint8)[54:].reshape(144, 176, 3)[::-1, :, ::-1]
        assert png.shape == (144, 176, 3) and np.array_equal(png, bmp)
        r = subprocess.run([str(MV), "-i", str(Path(d) / "in.264"), "-f", "bmp", "-o", str(Path(d) / "missing" / "dir")], capture_output=True, text=True)
        assert r.returncode != 0 and "cannot write" in r.stderr


@pytest.mark.gpu
def test_cli_2160p_distributed_extraction(cli):
    """BASELINE.json configs[4]: a 3840x2160 High-profile stream in 'distributed' extraction mode, through the
    CLI, against the files of the reference CLI (which may abort after writing them, see above)."""
    from minivideo_b200 import synth
    stream, _ = synth.generate(10, "2160p", seed=907)
    args = ["-f", "yuv420", "-n", "3", "-e", "distributed"]
    files, r = _run(MV, stream, args + ["-o", "."])
    assert r.returncode == 0, (r.stdout[-1500:], r.stderr[-1500:])
    got = {k: digest(v) for k, v in files.items()}
    want = _reference_files(stream, args, may_crash=True, keep=lambda data: len(data) == 3840 * 2160 * 3 // 2)
    assert set(want) <= set(got) and len(want) >= 2
    full = {k: v for k, v in want.items() if v is not None}      # a file cut short by the abort does not count
    assert len(full) >= 2
    for name in full:
        assert full[name] == got[name], name


@pytest.mark.gpu
def test_cli_all_gpus_writes_the_same_files_as_one_gpu(cli):
    """-d all: one feeder thread and context per GPU, batches dealt round-robin (SURVEY.md section 8e); the files
    do not depend on how many GPUs took part.  On a one-GPU box this still exercises the feeder path."""
    from minivideo_b200 import synth
    stream, _ = synth.generate(13, width_mbs=20, height_mbs=12, profile_idc=100, transform8x8=1, scaling_lists=1, seed=909)
    outs = []
    for dev in ("0", "all"):
        with tempfile.TemporaryDirectory(dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as d:
            (Path(d) / "in.264").write_bytes(stream)
            r = subprocess.run([str(MV), "-i", str(Path(d) / "in.264"), "-f", "bmp", "-n", "13", "-b", "2", "-d", dev, "-o", d],
                               capture_output=True, text=True)
            assert r.returncode == 0 and "13 picture(s) exported" in r.stdout, (r.stdout, r.stderr)
            outs.append({p.name: p.read_bytes() for p in Path(d).iterdir() if p.name != "in.264"})
    assert len(outs[0]) == 13 and outs[0] == outs[1]


@pytest.mark.gpu
@pytest.mark.parametrize("geometry_change", [False, True], ids=["same_size", "new_size"])
@pytest.mark.parametrize("fmt", ["yuv420", "bmp"])
def test_cli_follows_parameter_set_changes_like_the_reference_cli(cli, geometry_change, fmt):
    """A stream whose SPS / PPS change between pictures (other scaling lists, chroma QP offsets, pic_init_qp, and
    with `new_size` other picture dimensions): the reference re-decodes every parameter set where it meets it
    (h264.c:128-150); mvt_extract() switches tables -- and output size -- per parameter generation."""
    from helpers import paramset_change_stream
    stream, segs = paramset_change_stream(geometry_change)
    want, _ = _run_both(stream, ["-f", fmt, "-n", "6"])
    assert len(want) == 6
    for extra in ([], ["-b", "1"], ["-b", "4", "-t", "2"]):      # batches that end at, inside and across the segments
        _, got = _run_both(stream, ["-f", fmt, "-n", "6"] + extra)
        assert want == got, extra


@pytest.mark.gpu
def test_cli_skips_a_picture_it_cannot_decode_like_the_reference_cli(cli):
    """The reference counts a picture that fails and goes on (h264.c:103-109); the pictures after it move up one
    number (export.c:630 numbers by pictures decoded).  Picture 1 of 5 is turned into a P slice (slice_type 5), which
    both decoders refuse."""
    from helpers import PAD, split_nals
    from minivideo_b200 import synth
    stream, _ = synth.generate(5, width_mbs=6, height_mbs=4, profile_idc=100, transform8x8=1, seed=31)
    nals = split_nals(stream)
    bad = nals[3][:5] + bytes([0b10100000 | (nals[3][5] & 0x0f)]) + nals[3][6:]     # first_mb 0 ('1'), slice_type ue '010..'
    broken = b"".join(nals[:3] + [bad] + nals[4:]) + PAD
    good, _ = _run_both(stream, ["-f", "yuv420", "-n", "5"])
    want = _reference_files(broken, ["-f", "yuv420", "-n", "5"], may_crash=True)
    files, r = _run(MV, broken, ["-f", "yuv420", "-n", "5", "-o", "."])
    got = {k: digest(v) for k, v in files.items()}
    assert sorted(want) == sorted(got) == ["in_0.yuv", "in_1.yuv", "in_2.yuv", "in_3.yuv"]
    assert want == got
    assert got["in_0.yuv"] == good["in_0.yuv"] and got["in_1.yuv"] == good["in_2.yuv"] and got["in_3.yuv"] == good["in_4.yuv"]
    assert r.returncode == 1 and "4 of 5 pictures exported" in r.stderr and "picture 1 skipped" in r.stderr
