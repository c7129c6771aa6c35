"""The BMP / TGA writers of mv_thumbcore.c against the reference's own vendored writers (oracle/_ref/ref_png with a
format argument = stbi_write_bmp / stbi_write_tga of minivideo/src/stb_image_write.h, the calls export_idr_bmp() /
export_idr_tga() make, export.c:570,:601), on pictures built to hit the packet rules of the run-length TGA:
runs of exactly 128 / 129 / 256 pixels, alternating pixels (a raw packet gives its last pixel back when pixel k
equals pixel k-2), widths 1..3, rows that end inside a run."""
import ctypes as C
import subprocess
import tempfile
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
REF = ROOT / "oracle" / "_ref" / "ref_png"
FMT = {"bmp": 1, "tga": 2, "png": 3}                     # MVT_BMP, MVT_TGA, MVT_PNG (mv_thumbcore.h)


@pytest.fixture(scope="module")
def lib():
    from minivideo_b200 import build
    build.build_thumbnailer()
    lib = C.CDLL(str(ROOT / "minivideo_b200" / "libminivideo_b200.so"))
    lib.mvt_write_image.argtypes = [C.c_char_p, C.c_int, C.c_void_p, C.c_int, C.c_int]
    return lib


def pictures():
    rng = np.random.default_rng(5)

    def runs(lengths, w):
        px = np.concatenate([np.tile(rng.integers(0, 256, (1, 3)), (n, 1)) for n in lengths])
        h = -(-len(px) // w)
        px = np.concatenate([px, rng.integers(0, 256, (h * w - len(px), 3))])
        return px.reshape(h, w, 3)
    yield "runs-128-129-256", runs([128, 129, 256, 1, 2, 127, 300, 3], 473)
    yield "runs-across-rows", runs([500, 7, 130, 128, 128, 1], 131)
    ab = np.zeros((4, 300, 3), np.int64)
    ab[:, ::2] = (10, 20, 30)
    ab[:, 1::2] = (200, 100, 50)
    yield "alternating", ab
    aab = np.tile(np.array([[1, 2, 3], [1, 2, 3], [9, 8, 7]]), (100, 1)).reshape(1, 300, 3)
    yield "aab", np.tile(aab, (3, 1, 1))
    yield "noise", rng.integers(0, 256, (17, 259, 3))
    yield "few-colours", rng.integers(0, 2, (16, 400, 1)).repeat(3, 2) * 255
    for w in (1, 2, 3, 5):
        yield f"width-{w}", rng.integers(0, 3, (9, w, 3)) * 90
    yield "flat", np.full((5, 1000, 3), 77)


@pytest.mark.parametrize("fmt", ["bmp", "tga", "png"])
@pytest.mark.parametrize("name,img", list(pictures()), ids=[n for n, _ in pictures()])
def test_writer_files_equal_the_reference_writers(lib, fmt, name, img):
    from helpers import digest, reference_output
    img = np.ascontiguousarray(np.asarray(img) & 255, np.uint8)
    h, w, _ = img.shape

    def live():
        with tempfile.TemporaryDirectory() as d:
            img.tofile(Path(d) / "in.rgb")
            subprocess.run([str(REF), str(w), str(h), str(Path(d) / "in.rgb"), str(Path(d) / "want"), fmt], check=True)
            return digest((Path(d) / "want").read_bytes())
    want = reference_output(f"ref_png {fmt} {name}", live, REF.exists())
    with tempfile.TemporaryDirectory() as d:
        assert lib.mvt_write_image(str(Path(d) / "got").encode(), FMT[fmt], img.ctypes.data, w, h) == 1
        assert digest((Path(d) / "got").read_bytes()) == want


def test_writer_rejects_bad_arguments(lib):
    buf = np.zeros(48, np.uint8)
    assert lib.mvt_write_image(b"/nonexistent-dir/x.bmp", 1, buf.ctypes.data, 4, 4) == 0
    assert lib.mvt_write_image(b"/tmp/x.bmp", 1, buf.ctypes.data, 0, 4) == 0
    assert lib.mvt_write_image(b"/tmp/x.bmp", 9, buf.ctypes.data, 4, 4) == 0


def test_extract_rejects_bad_arguments_without_touching_a_gpu(lib):
    """mvt_extract(): argument checks come before any CUDA call."""
    from minivideo_b200 import synth
    stream, _ = synth.generate(2, "cif", seed=5)
    buf = np.frombuffer(stream, np.uint8)
    lib.mvt_extract.argtypes = [C.c_void_p, C.c_size_t, C.c_char_p, C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                C.c_int, C.c_int, C.POINTER(C.c_int)]
    n = C.c_int(7)
    ok = dict(fmt=0, n_want=1, mode=0, scale=1, device=0, threads=1, batch=0)
    for bad in (dict(fmt=9), dict(fmt=-1), dict(n_want=0), dict(scale=0), dict(batch=-1)):
        a = dict(ok, **bad)
        assert lib.mvt_extract(buf.ctypes.data, len(buf), b"x", b"/tmp", a["fmt"], a["n_want"], a["mode"], a["scale"],
                               a["device"], a["threads"], a["batch"], C.byref(n)) == 0, bad
        assert n.value == 0
    assert lib.mvt_extract(None, 0, b"x", b"/tmp", 0, 1, 0, 1, 0, 1, 0, C.byref(n)) == 0
    garbage = np.arange(4096, dtype=np.uint8)
    assert lib.mvt_extract(garbage.ctypes.data, len(garbage), b"x", b"/tmp", 0, 1, 0, 1, 0, 1, 0, C.byref(n)) == 0   # no SPS/PPS
