"""TEST INFRASTRUCTURE: ctypes binding of oracle/librecon_oracle.so (recon_oracle.c)."""
from __future__ import annotations

import ctypes as C
import subprocess
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
_LIB = None


class OracleSps(C.Structure):
    _fields_ = [("width_mbs", C.c_int32), ("height_mbs", C.c_int32),
                ("ls4", C.c_int32 * (3 * 6 * 16)), ("ls8", C.c_int32 * (6 * 64)),
                ("cb_qp_offset", C.c_int32), ("cr_qp_offset", C.c_int32)]


def lib():
    global _LIB
    if _LIB is None:
        so = HERE / "librecon_oracle.so"
        srcs = (HERE / "recon_oracle.c", HERE / "recon_oracle.h", HERE / "Makefile")
        if not so.exists() or any(so.stat().st_mtime < s.stat().st_mtime for s in srcs):
            subprocess.run(["make", "-C", str(HERE), "oracle"], check=True, capture_output=True)
        _LIB = C.CDLL(str(so))
        _LIB.oracle_chroma_qp.restype = C.c_int
    return _LIB


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def level_scale(lists4x4: np.ndarray | None, list8x8: np.ndarray | None):
    """(ls4[3,6,16], ls8[6,64]) from zig-zag scaling lists (intra Y,Cb,Cr 4x4; intra Y 8x8)."""
    ls4 = np.zeros((3, 6, 16), np.int32)
    ls8 = np.zeros((6, 64), np.int32)
    l4 = np.ascontiguousarray(lists4x4[:3], np.uint8) if lists4x4 is not None else None
    l8 = np.ascontiguousarray(list8x8, np.uint8) if list8x8 is not None else None
    lib().oracle_build_level_scale(_p(l4) if l4 is not None else None, _p(l8) if l8 is not None else None,
                                   _p(ls4), _p(ls8))
    return ls4, ls8


def make_sps(soa) -> OracleSps:
    ls4, ls8 = level_scale(soa.lists4x4, soa.lists8x8[0])
    s = OracleSps()
    s.width_mbs, s.height_mbs = soa.width_mbs, soa.height_mbs
    C.memmove(s.ls4, ls4.ctypes.data, ls4.nbytes)
    C.memmove(s.ls8, ls8.ctypes.data, ls8.nbytes)
    s.cb_qp_offset, s.cr_qp_offset = soa.cb_qp_offset, soa.cr_qp_offset
    return s


def reconstruct(soa, want_residual: bool = False):
    """Returns (yuv [P, 1.5*W*H] u8, residual [P*N,384] i16 | None)."""
    L = lib()
    sps = make_sps(soa)
    W, H, N = soa.width, soa.height, soa.n_mbs
    yuv = np.zeros((soa.n_pics, W * H * 3 // 2), np.uint8)
    res = np.zeros((soa.n_pics * N, 384), np.int16) if want_residual else None
    for p in range(soa.n_pics):
        s = slice(p * N, (p + 1) * N)
        kind = np.ascontiguousarray(soa.mb_kind[s]); i16 = np.ascontiguousarray(soa.i16_mode[s])
        cm = np.ascontiguousarray(soa.chroma_mode[s]); qp = np.ascontiguousarray(soa.qp_y[s])
        modes = np.ascontiguousarray(soa.luma_modes[s]); coeff = np.ascontiguousarray(soa.coeff[s])
        y = yuv[p, :W * H]; cb = yuv[p, W * H:W * H * 5 // 4]; cr = yuv[p, W * H * 5 // 4:]
        r = res[s] if want_residual else None
        L.oracle_reconstruct_picture(C.byref(sps), _p(kind), _p(i16), _p(cm), _p(qp), _p(modes), _p(coeff),
                                     _p(y), _p(cb), _p(cr), _p(r) if r is not None else None)
    return yuv, res


def yuv_to_rgb(yuv: np.ndarray, width: int, height: int, scale: int = 1) -> np.ndarray:
    """[P, 1.5*W*H] -> [P, H/s, W/s, 3]"""
    L = lib()
    P = yuv.shape[0]
    out = np.zeros((P, height // scale, width // scale, 3), np.uint8)
    for p in range(P):
        fr = np.ascontiguousarray(yuv[p])
        y = fr[:width * height]; cb = fr[width * height:width * height * 5 // 4]; cr = fr[width * height * 5 // 4:]
        L.oracle_yuv420_to_rgb(width, height, _p(y), _p(cb), _p(cr), scale, _p(out[p]))
    return out
