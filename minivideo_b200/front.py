"""ctypes mirror of include/mvfront.h (libmvfront.so): the host front end that turns a CAVLC intra stream,
Annex-B or in an MP4 / QuickTime file, into the mvgpu.h structure-of-arrays."""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import numpy as np

from .synth import Soa

_LIB = None


class Info(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "width_mbs", "height_mbs", "profile_idc", "level_idc", "n_idr", "transform_8x8_mode",
        "cb_qp_offset", "cr_qp_offset", "pic_init_qp", "crop_left", "crop_right", "crop_top", "crop_bottom")]
    _fields_ += [("level_scale4x4", C.c_int32 * 288), ("level_scale8x8", C.c_int32 * 384),
                 ("n_generations", C.c_int32), ("generation", C.c_int32)]


class FrontBatch(C.Structure):
    _fields_ = [("n_pics", C.c_int32), ("mb_kind", C.c_void_p), ("i16_mode", C.c_void_p),
                ("chroma_mode", C.c_void_p), ("qp_y", C.c_void_p), ("cbp", C.c_void_p),
                ("luma_modes", C.c_void_p), ("coeff", C.c_void_p), ("status", C.c_void_p)]


class FrontPackedBatch(C.Structure):
    """mvf_packed_batch of include/mvfront.h."""
    _fields_ = [("n_pics", C.c_int32), ("mb_kind", C.c_void_p), ("i16_mode", C.c_void_p),
                ("chroma_mode", C.c_void_p), ("qp_y", C.c_void_p), ("luma_modes", C.c_void_p),
                ("nz_blocks", C.c_void_p), ("word_off", C.c_void_p), ("pic_off", C.c_void_p),
                ("words", C.c_void_p), ("words_capacity", C.c_size_t), ("status", C.c_void_p),
                ("words_needed", C.c_size_t)]


class FrontError(RuntimeError):
    def __init__(self, msg, code):
        super().__init__(msg)
        self.code = code


def lib():
    global _LIB
    if _LIB is None:
        path = Path(__file__).resolve().parent / "libmvfront.so"
        if not path.exists():
            from . import build
            build.build_front()
        _LIB = C.CDLL(str(path))
        vp = C.c_void_p
        _LIB.mvf_open_annexb.argtypes = [vp, C.c_size_t, C.POINTER(vp)]
        _LIB.mvf_open_mp4.argtypes = [vp, C.c_size_t, C.POINTER(vp)]
        _LIB.mvf_close.argtypes = [vp]
        _LIB.mvf_last_error.argtypes = [vp]
        _LIB.mvf_last_error.restype = C.c_char_p
        _LIB.mvf_get_info.argtypes = [vp, C.POINTER(Info)]
        _LIB.mvf_select_idr.argtypes = [vp, C.c_int, C.c_int, vp]
        _LIB.mvf_parse_pictures.argtypes = [vp, vp, C.c_int, C.c_int, C.POINTER(FrontBatch), C.c_int]
        _LIB.mvf_parse_pictures_packed.argtypes = [vp, vp, C.c_int, C.c_int, C.POINTER(FrontPackedBatch), C.c_int]
        _LIB.mvf_generation_count.argtypes = [vp]
        _LIB.mvf_get_generation_info.argtypes = [vp, C.c_int, C.POINTER(Info)]
        _LIB.mvf_picture_generation.argtypes = [vp, C.c_int]
        _LIB.mvf_parser_create.argtypes = [vp, C.c_int, C.POINTER(vp)]
        _LIB.mvf_parser_destroy.argtypes = [vp]
        _LIB.mvf_parser_parse.argtypes = [vp, vp, C.c_int, C.c_int, C.POINTER(FrontBatch)]
        _LIB.mvf_parser_parse_packed.argtypes = [vp, vp, C.c_int, C.c_int, C.POINTER(FrontPackedBatch)]
        _LIB.mvf_parser_last_error.argtypes = [vp]
        _LIB.mvf_parser_last_error.restype = C.c_char_p
    return _LIB


class Stream:
    """An opened stream (mvf_stream): an Annex-B byte stream (mvf_open_annexb) or an MP4 / QuickTime file
    (container="mp4", mvf_open_mp4)."""

    def __init__(self, data: bytes, container: str = "annexb"):
        self._lib = lib()
        opener = {"annexb": self._lib.mvf_open_annexb, "mp4": self._lib.mvf_open_mp4}.get(container)
        if opener is None:
            raise ValueError(f"container must be 'annexb' or 'mp4', not {container!r}")
        self._buf = np.frombuffer(data, np.uint8)          # keeps the bytes alive
        self.handle = C.c_void_p()
        rc = opener(self._buf.ctypes.data, len(data), C.byref(self.handle))
        if rc != 1:
            raise FrontError(self._lib.mvf_last_error(None).decode(), rc)
        self.info = Info()
        self._lib.mvf_get_info(self.handle, C.byref(self.info))

    def close(self):
        if self.handle:
            self._lib.mvf_close(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def n_idr(self):
        return self.info.n_idr

    @property
    def n_generations(self):
        return self._lib.mvf_generation_count(self.handle)

    def generation_info(self, gen: int) -> "Info":
        out = Info()
        if self._lib.mvf_get_generation_info(self.handle, gen, C.byref(out)) != 1:
            raise FrontError(f"no parameter generation {gen}", 0)
        return out

    def picture_generations(self) -> np.ndarray:
        """Per IDR picture the index of its parameter generation (-1: no usable SPS/PPS)."""
        return np.array([self._lib.mvf_picture_generation(self.handle, i) for i in range(self.n_idr)], np.int32)

    def level_scale(self, info: "Info | None" = None):
        info = info or self.info
        return (np.array(info.level_scale4x4, np.int32).reshape(3, 6, 16),
                np.array(info.level_scale8x8, np.int32).reshape(6, 64))

    def select_idr(self, n_wanted: int, mode: int) -> np.ndarray:
        out = np.zeros(max(n_wanted, 1), np.int32)
        n = self._lib.mvf_select_idr(self.handle, n_wanted, mode, out.ctypes.data)
        return out[:n]

    def _info_for(self, first, indices):
        """mvf_info of the generation the first requested picture belongs to."""
        i0 = int(indices[0]) if indices is not None and len(indices) else first
        g = self._lib.mvf_picture_generation(self.handle, i0) if 0 <= i0 < self.n_idr else 0
        return self.generation_info(max(g, 0))

    def parse(self, first: int = 0, count: int | None = None, indices=None, n_threads: int | None = None,
              arrays: dict | None = None, tolerant: bool = False) -> Soa:
        """CAVLC-parse pictures into a Soa (numpy arrays, or caller-provided `arrays`).  tolerant=True: failed
        pictures are reported in soa.status (one code per picture) instead of failing the call."""
        if indices is not None:
            indices = np.ascontiguousarray(indices, np.int32)
            count = len(indices)
        elif count is None:
            count = self.n_idr - first
        info = self._info_for(first, indices)
        n = info.width_mbs * info.height_mbs * count
        a = arrays or dict(mb_kind=np.zeros(n, np.uint8), i16_mode=np.zeros(n, np.uint8), chroma_mode=np.zeros(n, np.uint8),
                           qp_y=np.zeros(n, np.int8), cbp=np.zeros(n, np.uint8), luma_modes=np.zeros((n, 16), np.uint8),
                           coeff=np.zeros((n, 384), np.int16))
        status = np.zeros(max(count, 1), np.int32) if tolerant else None
        b = FrontBatch(count, *(a[k].ctypes.data for k in ("mb_kind", "i16_mode", "chroma_mode", "qp_y", "cbp", "luma_modes", "coeff")),
                       status.ctypes.data if tolerant else None)
        rc = self._lib.mvf_parse_pictures(self.handle, indices.ctypes.data if indices is not None else None, first, count,
                                          C.byref(b), n_threads or os.cpu_count() or 1)
        if rc != 1:
            raise FrontError(self._lib.mvf_last_error(self.handle).decode(), rc)
        soa = Soa(info.width_mbs, info.height_mbs, count, a["mb_kind"], a["i16_mode"], a["chroma_mode"],
                  a["qp_y"], a["cbp"], a["luma_modes"], a["coeff"],
                  cb_qp_offset=info.cb_qp_offset, cr_qp_offset=info.cr_qp_offset)
        soa.status = status[:count] if tolerant else None
        return soa

    def parse_packed(self, first: int = 0, count: int | None = None, indices=None, n_threads: int | None = None,
                     words_capacity: int | None = None) -> dict:
        """CAVLC-parse pictures straight into the packed transfer format (mvf_parse_pictures_packed).
        Returns the arrays of mvg_packed_batch as a dict (plus n_pics, n_mbs)."""
        if indices is not None:
            indices = np.ascontiguousarray(indices, np.int32)
            count = len(indices)
        elif count is None:
            count = self.n_idr - first
        info = self._info_for(first, indices)
        N = info.width_mbs * info.height_mbs
        n = N * count
        cap = words_capacity if words_capacity is not None else n * 408
        a = dict(mb_kind=np.zeros(n, np.uint8), i16_mode=np.zeros(n, np.uint8), chroma_mode=np.zeros(n, np.uint8),
                 qp_y=np.zeros(n, np.int8), luma_modes=np.zeros((n, 16), np.uint8), nz_blocks=np.zeros(n, np.uint32),
                 word_off=np.zeros(n, np.uint32), pic_off=np.zeros(count + 1, np.uint64), words=np.zeros(max(cap, 1), np.uint16))
        b = FrontPackedBatch(count, *(a[k].ctypes.data for k in ("mb_kind", "i16_mode", "chroma_mode", "qp_y", "luma_modes",
                                                                  "nz_blocks", "word_off", "pic_off", "words")), cap)
        rc = self._lib.mvf_parse_pictures_packed(self.handle, indices.ctypes.data if indices is not None else None, first,
                                                 count, C.byref(b), n_threads or os.cpu_count() or 1)
        if rc != 1:
            raise FrontError(self._lib.mvf_last_error(self.handle).decode(), rc)
        a["words"] = a["words"][: max(int(a["pic_off"][count]), 1)]
        a["n_pics"], a["n_mbs"] = count, N
        return a
