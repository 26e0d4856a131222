"""ORACLE -- test infrastructure only.

ctypes front-ends for (a) ``port``: our plain-C restatement (``himg_oracle.c``) and (b) ``ref``:
the unmodified reference compiled into ``oracle/_ref/libhimg_ref.so`` (present when it was built
in the container that has ``/root/reference``; it travels to the GPU box with the snapshot).

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline / ``--impl reference``
leg may import this package.  The product package ``himg_b200`` never does.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import build_oracle

_u8p = C.POINTER(C.c_uint8)
_i16p = C.POINTER(C.c_int16)
_u16p = C.POINTER(C.c_uint16)
_u32p = C.POINTER(C.c_uint32)
_ip = C.POINTER(C.c_int)


def _p(a: np.ndarray, t=_u8p):
    return a.ctypes.data_as(t)


def _u8(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.uint8)


class _Port:
    """The plain-C restatement."""

    def __init__(self):
        path = build_oracle.build_port()
        self.lib = L = C.CDLL(path)
        L.ho_fnv1a64.restype = C.c_uint64
        L.ho_fnv1a64.argtypes = [_u8p, C.c_size_t]
        L.ho_synth_image.argtypes = [_u8p, C.c_int, C.c_int, C.c_int, C.c_uint32, C.c_uint32]
        L.ho_synth_image.restype = None
        # (sizes of images, streams and buffers are 64-bit: they may exceed 2 GiB)
        L.ho_encode_bound.restype = C.c_size_t
        L.ho_encode_bound.argtypes = [C.c_int, C.c_int, C.c_int]
        L.ho_encode.restype = C.c_longlong
        L.ho_encode.argtypes = [_u8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _u8p, C.c_size_t]
        L.ho_decode.argtypes = [_u8p, C.c_size_t, C.c_int, _u8p, C.c_size_t, _ip, _ip, _ip]
        L.ho_huff_compress.restype = C.c_longlong
        L.ho_huff_compress.argtypes = [_u8p, C.c_size_t, _u8p, C.c_size_t, C.c_size_t]
        L.ho_huff_uncompress.argtypes = [_u8p, C.c_size_t, C.c_size_t, C.c_int, _u8p, C.c_size_t, C.c_int, C.c_size_t]
        L.ho_huff_histogram.argtypes = [_u8p, C.c_size_t, C.c_size_t, _u32p]
        L.ho_huff_histogram.restype = None
        L.ho_huff_tree.argtypes = [_u32p, C.c_int, _u32p, _u8p, _u8p]
        L.ho_shift_table.argtypes = [C.c_int, C.c_int, _u8p]
        L.ho_shift_table.restype = None
        L.ho_lowres_map_table.argtypes = [C.c_int, _u16p]
        L.ho_lowres_map_table.restype = None
        L.ho_fullres_map_table.argtypes = [_u16p]
        L.ho_fullres_map_table.restype = None
        L.ho_map_to_8bit.argtypes = [_u16p, C.c_int]
        L.ho_mapfun_serialize.argtypes = [_u16p, _u8p]
        L.ho_mapfun_parse.argtypes = [_u8p, C.c_int, _i16p]
        L.ho_rgb_to_ycbcr.argtypes = [_u8p, _u8p, C.c_int, C.c_int, C.c_int, C.c_int]
        L.ho_rgb_to_ycbcr.restype = None
        L.ho_ycbcr_to_rgb.argtypes = [_u8p, C.c_int, C.c_int, C.c_int]
        L.ho_ycbcr_to_rgb.restype = None
        L.ho_lowres_sample.argtypes = [_u8p, C.c_int, C.c_int, C.c_int, _u8p]
        L.ho_lowres_sample.restype = None
        L.ho_lowres_encode.argtypes = [_u8p, C.c_int, C.c_int, _u16p, _u8p]
        L.ho_lowres_encode.restype = None
        L.ho_lowres_decode.argtypes = [_u8p, C.c_int, C.c_int, _i16p, _u8p]
        L.ho_lowres_decode.restype = None
        L.ho_lowres_block.argtypes = [_u8p, C.c_int, C.c_int, C.c_int, C.c_int, _i16p]
        L.ho_lowres_block.restype = None
        L.ho_wht_forward.argtypes = [_i16p, _i16p]
        L.ho_wht_forward.restype = None
        L.ho_wht_inverse.argtypes = [_i16p, _i16p]
        L.ho_wht_inverse.restype = None
        L.ho_fullres_planes.argtypes = [_u8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _u8p, _u8p, _u8p, _u16p, _u8p]
        L.ho_fullres_planes.restype = None
        L.ho_fullres_restore.argtypes = [_u8p, C.c_int, C.c_int, C.c_int, C.c_int, _u8p, _u8p, _u8p, _i16p, _u8p]
        L.ho_fullres_restore.restype = None

    # -- helpers ---------------------------------------------------------------------------
    def fnv(self, a) -> int:
        a = _u8(a).reshape(-1)
        return int(self.lib.ho_fnv1a64(_p(a), a.size))

    def synth(self, w, h, nch, seed=1, amp=6) -> np.ndarray:
        out = np.empty((h, w, nch), np.uint8)
        self.lib.ho_synth_image(_p(out), w, h, nch, seed, amp)
        return out

    # -- whole codec -----------------------------------------------------------------------
    def encode_bound(self, w, h, nch) -> int:
        return int(self.lib.ho_encode_bound(w, h, nch))

    def encode(self, img, quality=50, use_ycbcr=True, pixel_stride=None, w=None, h=None, nch=None) -> bytes:
        img = _u8(img)
        if w is None:
            h, w, nch = img.shape
        ps = pixel_stride or nch
        out = np.empty(self.encode_bound(w, h, nch), np.uint8)
        n = self.lib.ho_encode(_p(img), w, h, ps, nch, quality, int(use_ycbcr), _p(out), out.size)
        if n <= 0:
            raise RuntimeError("oracle encode failed")
        return out[:n].tobytes()

    def decode(self, data: bytes, strict=True):
        buf = np.frombuffer(data, np.uint8)
        w, h, n = C.c_int(), C.c_int(), C.c_int()
        cap = 1 << 16
        while True:
            out = np.empty(cap, np.uint8)
            r = self.lib.ho_decode(_p(buf), buf.size, int(strict), _p(out), cap, C.byref(w), C.byref(h), C.byref(n))
            if r == -1:
                cap = w.value * h.value * n.value
                continue
            if r == 0:
                return None
            img = out[: w.value * h.value * n.value].reshape(h.value, w.value, n.value)
            return img if img.size == cap else img.copy()

    # -- stages ----------------------------------------------------------------------------
    def shift_table(self, quality, chroma) -> np.ndarray:
        out = np.empty(64, np.uint8)
        self.lib.ho_shift_table(quality, int(chroma), _p(out))
        return out

    def lowres_map_table(self, quality) -> np.ndarray:
        t = np.empty(128, np.uint16)
        self.lib.ho_lowres_map_table(quality, _p(t, _u16p))
        return t

    def fullres_map_table(self) -> np.ndarray:
        t = np.empty(128, np.uint16)
        self.lib.ho_fullres_map_table(_p(t, _u16p))
        return t

    def map_to_8bit(self, table, x) -> int:
        t = np.ascontiguousarray(table, np.uint16)
        return int(self.lib.ho_map_to_8bit(_p(t, _u16p), int(x)))

    def mapfun_serialize(self, table) -> bytes:
        t = np.ascontiguousarray(table, np.uint16)
        out = np.empty(256, np.uint8)
        n = self.lib.ho_mapfun_serialize(_p(t, _u16p), _p(out))
        return out[:n].tobytes()

    def mapfun_parse(self, data: bytes):
        buf = np.frombuffer(data, np.uint8)
        un = np.empty(256, np.int16)
        ok = self.lib.ho_mapfun_parse(_p(buf), buf.size, _p(un, _i16p))
        return un if ok else None

    def rgb_to_ycbcr(self, img) -> np.ndarray:
        img = _u8(img)
        h, w, n = img.shape
        out = np.empty_like(img)
        self.lib.ho_rgb_to_ycbcr(_p(img), _p(out), w, h, n, n)
        return out

    def ycbcr_to_rgb(self, img) -> np.ndarray:
        out = _u8(img).copy()
        h, w, n = out.shape
        self.lib.ho_ycbcr_to_rgb(_p(out), w, h, n)
        return out

    def lowres_sample(self, cm) -> np.ndarray:
        """cm: colour-mapped [h][w][nch] -> L [nch][rows][cols]."""
        cm = _u8(cm)
        h, w, n = cm.shape
        rows, cols = (h + 7) >> 3, (w + 7) >> 3
        L = np.empty((n, rows, cols), np.uint8)
        flat = cm.reshape(-1)
        for c in range(n):
            self.lib.ho_lowres_sample(_p(flat[c:]), n, w, h, _p(L[c]))
        return L

    def lowres_channel_size(self, rows, cols) -> int:
        return ((rows + 15) // 16) * ((cols + 15) // 16) + rows * cols

    def lowres_encode(self, L, quality) -> np.ndarray:
        """L [nch][rows][cols] -> LRES unpacked bytes (all channels back to back)."""
        L = _u8(L)
        n, rows, cols = L.shape
        lt = self.lowres_map_table(quality)
        sz = self.lowres_channel_size(rows, cols)
        out = np.empty((n, sz), np.uint8)
        for c in range(n):
            self.lib.ho_lowres_encode(_p(L[c]), rows, cols, _p(lt, _u16p), _p(out[c]))
        return out.reshape(-1)

    def lowres_decode(self, lres, nch, rows, cols, unmap) -> np.ndarray:
        lres = _u8(lres).reshape(nch, -1)
        un = np.ascontiguousarray(unmap, np.int16)
        R = np.zeros((nch, rows, cols), np.uint8)
        for c in range(nch):
            row = np.ascontiguousarray(lres[c])
            self.lib.ho_lowres_decode(_p(row), rows, cols, _p(un, _i16p), _p(R[c]))
        return R

    def fullres_planes(self, cm, L, quality, ycbcr) -> np.ndarray:
        cm = _u8(cm)
        L = _u8(L)
        h, w, n = cm.shape
        rows, cols = (h + 7) >> 3, (w + 7) >> 3
        sl, sc = self.shift_table(quality, 0), self.shift_table(quality, 1)
        ft = self.fullres_map_table()
        out = np.empty(rows * cols * 64 * n, np.uint8)
        self.lib.ho_fullres_planes(_p(cm), w, h, n, n, int(ycbcr), _p(L), _p(sl), _p(sc), _p(ft, _u16p), _p(out))
        return out

    def fullres_restore(self, planes, w, h, nch, ycbcr, R, shift_luma, shift_chroma, unmap) -> np.ndarray:
        planes = _u8(planes)
        R = _u8(R)
        sl, sc = _u8(shift_luma), _u8(shift_chroma)
        un = np.ascontiguousarray(unmap, np.int16)
        out = np.empty((h, w, nch), np.uint8)
        self.lib.ho_fullres_restore(_p(planes), w, h, nch, int(ycbcr), _p(R), _p(sl), _p(sc), _p(un, _i16p), _p(out))
        return out

    def wht_forward(self, blk) -> np.ndarray:
        a = np.ascontiguousarray(blk, np.int16).reshape(64)
        o = np.empty(64, np.int16)
        self.lib.ho_wht_forward(_p(a, _i16p), _p(o, _i16p))
        return o

    def wht_inverse(self, blk) -> np.ndarray:
        a = np.ascontiguousarray(blk, np.int16).reshape(64)
        o = np.empty(64, np.int16)
        self.lib.ho_wht_inverse(_p(a, _i16p), _p(o, _i16p))
        return o

    def huff_histogram(self, data, block_size=0) -> np.ndarray:
        d = _u8(data).reshape(-1)
        h = np.zeros(261, np.uint32)
        self.lib.ho_huff_histogram(_p(d), d.size, block_size, _p(h, _u32p))
        return h

    def huff_tree(self, hist, fast=False):
        h = np.ascontiguousarray(hist, np.uint32)
        code = np.zeros(261, np.uint32)
        ln = np.zeros(261, np.uint8)
        tree = np.zeros(360, np.uint8)
        bits = self.lib.ho_huff_tree(_p(h, _u32p), int(fast), _p(code, _u32p), _p(ln), _p(tree))
        return bits, code, ln, tree[: (max(bits, 0) + 7) // 8].tobytes()

    def huff_compress(self, data, block_size=0) -> bytes:
        d = _u8(data).reshape(-1)
        out = np.empty(2 * d.size + 4096, np.uint8)
        n = self.lib.ho_huff_compress(_p(out), out.size, _p(d), d.size, block_size)
        if n < 0:
            raise RuntimeError("oracle huff_compress overflow")
        return out[:n].tobytes()

    def huff_uncompress(self, data: bytes, out_size, block_size=0, block_no=-1, strict=True, unpacked_total=0):
        buf = np.frombuffer(data, np.uint8)
        out = np.empty(out_size, np.uint8)
        ok = self.lib.ho_huff_uncompress(_p(buf), buf.size, block_size, block_no, _p(out), out_size, int(strict), unpacked_total)
        return out if ok else None


class _Ref:
    """The unmodified reference, compiled in place (oracle/_ref/libhimg_ref.so)."""

    def __init__(self):
        path = build_oracle.build_ref()
        if not path or not os.path.exists(path):
            raise FileNotFoundError("oracle/_ref/libhimg_ref.so is not available")
        self.lib = L = C.CDLL(path)
        L.ref_encode.argtypes = [_u8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _u8p, C.c_int]
        L.ref_decode.argtypes = [_u8p, C.c_int, C.c_int, _u8p, C.c_int, _ip, _ip, _ip]
        L.ref_huff_compress.argtypes = [_u8p, _u8p, C.c_int, C.c_int]
        L.ref_huff_uncompress.argtypes = [_u8p, C.c_int, C.c_int, C.c_int, _u8p, C.c_int]
        L.ref_lowres_channel.argtypes = [_u8p, C.c_int, C.c_int, C.c_int, C.c_int, _u8p, _u8p]
        L.ref_lowres_restore.argtypes = [_u8p, C.c_int, C.c_int, _u8p, C.c_int, _u8p]
        L.ref_lowres_restore.restype = None
        L.ref_lowres_mapfun.argtypes = [C.c_int, _u8p]
        L.ref_lowres_mapfun.restype = None
        L.ref_fullres_mapfun.argtypes = [_u8p, C.c_int]
        L.ref_map_to_8bit.argtypes = [C.c_int, C.c_int, C.c_int]
        L.ref_quant_config.argtypes = [C.c_int, C.c_int, _u8p]
        L.ref_quant_pack.argtypes = [C.c_int, C.c_int, _i16p, _u8p]
        L.ref_quant_pack.restype = None
        L.ref_quant_unpack.argtypes = [C.c_int, C.c_int, _u8p, _i16p]
        L.ref_quant_unpack.restype = None
        L.ref_hadamard_forward.argtypes = [_i16p, _i16p]
        L.ref_hadamard_forward.restype = None
        L.ref_hadamard_inverse.argtypes = [_i16p, _i16p]
        L.ref_hadamard_inverse.restype = None
        L.ref_rgb_to_ycbcr.argtypes = [_u8p, _u8p, C.c_int, C.c_int, C.c_int, C.c_int]
        L.ref_rgb_to_ycbcr.restype = None
        L.ref_ycbcr_to_rgb.argtypes = [_u8p, C.c_int, C.c_int, C.c_int]
        L.ref_ycbcr_to_rgb.restype = None

    def encode(self, img, quality=50, use_ycbcr=True, pixel_stride=None, w=None, h=None, nch=None) -> bytes:
        img = _u8(img)
        if w is None:
            h, w, nch = img.shape
        ps = pixel_stride or nch
        rows, cols = (h + 7) >> 3, (w + 7) >> 3
        cap = 4096 + 2 * 360 + (rows * cols * 65 + 64) * nch
        out = np.empty(cap, np.uint8)
        n = self.lib.ref_encode(_p(img), w, h, ps, nch, quality, int(use_ycbcr), _p(out), cap)
        if n <= 0:
            raise RuntimeError("reference encode failed")
        return out[:n].tobytes()

    def decode(self, data: bytes, max_threads=1):
        """One worker thread by default: with max_threads=0 (hardware concurrency) the reference's
        decoder crashes intermittently on images with fewer block rows than threads (observed on
        520x24: 2 segfaults in 25 runs, none with one thread; decoder.cpp:274-329)."""
        buf = np.frombuffer(data, np.uint8)
        w, h, n = C.c_int(), C.c_int(), C.c_int()
        cap = 1 << 16
        while True:
            out = np.empty(cap, np.uint8)
            r = self.lib.ref_decode(_p(buf), buf.size, max_threads, _p(out), cap, C.byref(w), C.byref(h), C.byref(n))
            if r == -1:
                cap = w.value * h.value * n.value
                continue
            if r == 0:
                return None
            return out[: w.value * h.value * n.value].reshape(h.value, w.value, n.value).copy()

    def huff_compress(self, data, block_size=0) -> bytes:
        d = _u8(data).reshape(-1)
        out = np.zeros(d.size + 4096, np.uint8)
        n = self.lib.ref_huff_compress(_p(out), _p(d), d.size, block_size)
        return out[:n].tobytes()

    def huff_uncompress(self, data: bytes, out_size, block_size=0, block_no=-1):
        # the reference peeks one byte past a segment: keep slack after the buffer
        buf = np.concatenate([np.frombuffer(data, np.uint8), np.zeros(8, np.uint8)])
        out = np.empty(out_size + 8, np.uint8)
        ok = self.lib.ref_huff_uncompress(_p(buf), buf.size - 8, block_size, block_no, _p(out), out_size)
        return out[:out_size] if ok else None

    def lowres_channel(self, cm, chan, quality):
        cm = _u8(cm)
        h, w, n = cm.shape
        rows, cols = (h + 7) >> 3, (w + 7) >> 3
        L = np.empty((rows, cols), np.uint8)
        bd = np.empty(((rows + 15) // 16) * ((cols + 15) // 16) + rows * cols, np.uint8)
        flat = cm.reshape(-1)
        self.lib.ref_lowres_channel(_p(flat[chan:]), n, w, h, quality, _p(L), _p(bd))
        return L, bd

    def lowres_restore(self, blockdata, rows, cols, lmap: bytes) -> np.ndarray:
        bd = _u8(blockdata)
        lm = np.frombuffer(lmap, np.uint8)
        R = np.empty((rows, cols), np.uint8)
        self.lib.ref_lowres_restore(_p(bd), rows, cols, _p(lm), lm.size, _p(R))
        return R

    def lowres_mapfun(self, quality) -> bytes:
        out = np.empty(128, np.uint8)
        self.lib.ref_lowres_mapfun(quality, _p(out))
        return out.tobytes()

    def fullres_mapfun(self) -> bytes:
        out = np.empty(256, np.uint8)
        n = self.lib.ref_fullres_mapfun(_p(out), 256)
        return out[:n].tobytes()

    def map_to_8bit(self, which, quality, x) -> int:
        return int(self.lib.ref_map_to_8bit(which, quality, x)) & 0xFF

    def quant_config(self, quality, has_chroma) -> bytes:
        out = np.empty(64, np.uint8)
        n = self.lib.ref_quant_config(quality, int(has_chroma), _p(out))
        return out[:n].tobytes()

    def quant_pack(self, quality, chroma, blk) -> np.ndarray:
        a = np.ascontiguousarray(blk, np.int16).reshape(64)
        o = np.empty(64, np.uint8)
        self.lib.ref_quant_pack(quality, int(chroma), _p(a, _i16p), _p(o))
        return o

    def quant_unpack(self, quality, chroma, codes) -> np.ndarray:
        a = _u8(codes).reshape(64)
        o = np.empty(64, np.int16)
        self.lib.ref_quant_unpack(quality, int(chroma), _p(a), _p(o, _i16p))
        return o

    def hadamard_forward(self, blk) -> np.ndarray:
        a = np.ascontiguousarray(blk, np.int16).reshape(64)
        o = np.empty(64, np.int16)
        self.lib.ref_hadamard_forward(_p(a, _i16p), _p(o, _i16p))
        return o

    def hadamard_inverse(self, blk) -> np.ndarray:
        a = np.ascontiguousarray(blk, np.int16).reshape(64)
        o = np.empty(64, np.int16)
        self.lib.ref_hadamard_inverse(_p(a, _i16p), _p(o, _i16p))
        return o

    def rgb_to_ycbcr(self, img) -> np.ndarray:
        img = _u8(img)
        h, w, n = img.shape
        out = np.empty_like(img)
        self.lib.ref_rgb_to_ycbcr(_p(img), _p(out), w, h, n, n)
        return out

    def ycbcr_to_rgb(self, img) -> np.ndarray:
        out = _u8(img).copy()
        h, w, n = out.shape
        self.lib.ref_ycbcr_to_rgb(_p(out), w, h, n)
        return out


_port = None
_ref = None


def port() -> _Port:
    global _port
    if _port is None:
        _port = _Port()
    return _port


def ref_available() -> bool:
    try:
        ref()
        return True
    except (FileNotFoundError, OSError, RuntimeError):
        return False


def ref() -> _Ref:
    global _ref
    if _ref is None:
        _ref = _Ref()
    return _ref
