"""mv_png.c (RGB24 -> PNG) against the reference's own vendored writer (oracle/_ref/ref_png = stbi_write_png of
minivideo/src/stb_image_write.h, the call export_idr_png() makes, export.c:539): byte for byte, plus an
independent check that the file is a valid PNG holding the same pixels (zlib inflate + unfilter in numpy)."""
import ctypes as C
import subprocess
import tempfile
from pathlib import Path

import numpy as np
import pytest

from helpers import digest, reference_output
from helpers import png_decode as decode

ROOT = Path(__file__).resolve().parent.parent
REF_PNG = ROOT / "oracle" / "_ref" / "ref_png"


@pytest.fixture(scope="module")
def lib():
    from minivideo_b200 import build
    build.build_thumbnailer()
    lib = C.CDLL(str(ROOT / "minivideo_b200" / "libminivideo_b200.so"))
    lib.mvt_png_encode.restype = C.c_void_p
    lib.mvt_png_encode.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_size_t)]
    lib.free.argtypes = [C.c_void_p]
    return lib


def encode(lib, img: np.ndarray) -> bytes:
    img = np.ascontiguousarray(img, np.uint8)
    h, w, _ = img.shape
    n = C.c_size_t()
    p = lib.mvt_png_encode(img.ctypes.data, w, h, C.byref(n))
    assert p
    out = C.string_at(p, n.value)
    lib.free(p)
    return out


def reference(img: np.ndarray) -> bytes:
    h, w, _ = img.shape
    with tempfile.TemporaryDirectory() as d:
        np.ascontiguousarray(img, np.uint8).tofile(Path(d) / "in.rgb")
        subprocess.run([str(REF_PNG), str(w), str(h), str(Path(d) / "in.rgb"), str(Path(d) / "out.png")], check=True)
        return (Path(d) / "out.png").read_bytes()


def pictures():
    rng = np.random.default_rng(20)
    yield "1x1", rng.integers(0, 256, (1, 1, 3))
    yield "1x7", rng.integers(0, 256, (7, 1, 3))
    yield "5x1", rng.integers(0, 256, (1, 5, 3))
    yield "flat", np.full((32, 48, 3), 131)
    yield "noise", rng.integers(0, 256, (40, 56, 3))
    yy, xx = np.mgrid[0:96, 0:160]
    yield "gradient", np.stack([xx, yy * 2, (xx + yy) // 2], -1) & 255
    blocks = rng.integers(0, 256, (12, 20, 3)).repeat(8, 0).repeat(8, 1)
    yield "blocks", blocks
    yield "blocks+noise", (blocks + rng.integers(0, 3, blocks.shape)) & 255
    # long exact repeats: matches of 258, distances near the 32 K window, full hash buckets
    tile = rng.integers(0, 256, (3, 1100, 3))
    yield "repeat", np.tile(tile, (12, 1, 1))
    stripes = np.zeros((64, 4000, 3), np.int64)
    stripes[:, ::7] = 200
    stripes[::5] += 17
    yield "stripes", stripes & 255
    yield "few colours", rng.integers(0, 4, (120, 200, 3)) * 60


@pytest.mark.parametrize("name,img", list(pictures()), ids=[n for n, _ in pictures()])
def test_png_bytes_equal_the_reference_writer(lib, name, img):
    img = np.asarray(img, np.uint8)
    want = reference_output(f"ref_png {name}", lambda: digest(reference(img)), REF_PNG.exists())
    assert digest(encode(lib, img)) == want


@pytest.mark.parametrize("name,img", [p for p in pictures() if p[0] in ("1x1", "noise", "blocks+noise", "repeat")],
                         ids=["1x1", "noise", "blocks+noise", "repeat"])
def test_png_is_a_valid_file_holding_the_same_pixels(lib, name, img):
    img = np.asarray(img, np.uint8)
    assert np.array_equal(decode(encode(lib, img)), img)


def test_png_rejects_bad_arguments(lib):
    n = C.c_size_t(5)
    assert not lib.mvt_png_encode(None, 4, 4, C.byref(n)) and n.value == 0
    buf = np.zeros(48, np.uint8)
    assert not lib.mvt_png_encode(buf.ctypes.data, 0, 4, C.byref(n))
    assert not lib.mvt_png_encode(buf.ctypes.data, 4, -1, C.byref(n))


def test_png_random_small_images_equal_the_reference_writer(lib):
    """Sizes 1..40 and contents from flat to noise, with repeats at random distances: the corner cases of the
    filter choice (ties, first row) and of the match finder (matches at the very end, overlapping matches,
    the lazy step) show up in small pictures far more often than in large ones."""
    rng = np.random.default_rng(77)
    cases = []
    for k in range(60):
        w, h = int(rng.integers(1, 41)), int(rng.integers(1, 41))
        kind = k % 4
        if kind == 0:
            img = rng.integers(0, 256, (h, w, 3))
        elif kind == 1:
            img = rng.integers(0, 3, (h, w, 3)) * 100
        elif kind == 2:
            base = rng.integers(0, 256, (int(rng.integers(1, 5)), int(rng.integers(1, 7)), 3))
            img = np.tile(base, (h // base.shape[0] + 1, w // base.shape[1] + 1, 1))[:h, :w]
        else:
            yy, xx = np.mgrid[0:h, 0:w]
            img = np.stack([xx * 7 + yy, xx + yy * 5, (xx * yy) % 17], -1) + rng.integers(0, 2, (h, w, 3))
        cases.append((k, w, h, kind, np.asarray(img & 255, np.uint8)))
    want = reference_output("ref_png random_small", lambda: [digest(reference(c[-1])) for c in cases], REF_PNG.exists())
    for (k, w, h, kind, img), d in zip(cases, want, strict=True):
        assert digest(encode(lib, img)) == d, (k, w, h, kind)
