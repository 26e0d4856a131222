"""himg_b200 -- B200-native HIMG encode/decode hot path.

Python mirror of the reference's operator interface (himg::Encoder / himg::Decoder,
src/lib/encoder.h:20-64, src/lib/decoder.h:22-67) on top of the C ABI in include/himg_cuda.h.
PyTorch is only used for device memory, streams and torch.distributed; the codec itself is the
hand-written sm_100a CUDA in himg_b200/csrc.  There is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _native
from ._native import HimgError, LENIENT, STRICT  # noqa: F401

__all__ = ["Context", "Encoder", "Decoder", "HimgError", "STRICT", "LENIENT", "encode_bound", "fnv1a64"]


def encode_bound(w: int, h: int, nch: int) -> int:
    return int(_native.load().himgcu_encode_bound(w, h, nch))


def fnv1a64(data) -> int:
    """FNV-1a 64 of a bytes object / contiguous uint8 numpy array (SURVEY.md Appendix B checksum)."""
    buf = np.frombuffer(data, np.uint8) if isinstance(data, (bytes, bytearray, memoryview)) else np.ascontiguousarray(data, np.uint8)
    return int(_native.load().himgcu_fnv1a64(buf.ctypes.data, buf.size))


def _ptr(x):
    """Raw address of a numpy array (host) or a torch tensor (host or device)."""
    if x is None:
        return None
    if isinstance(x, np.ndarray):
        return x.ctypes.data
    return x.data_ptr()


class Context:
    """Owns device scratch and a stream on one GPU (himgcu_ctx)."""

    def __init__(self, device: int = 0, stream=None):
        self.lib = _native.load()
        h = C.c_void_p()
        rc = self.lib.himgcu_create(device, C.byref(h))
        if rc != _native.OK:
            raise HimgError(rc, f"cannot create a context on CUDA device {device} (no CPU fallback)")
        self.h = h
        self.device = device
        self._explicit_stream = False  # set_stream() was called by the user
        self._bound = None             # handle of the torch stream the tensor calls were last bound to
        if stream is not None:
            self.set_stream(stream)

    def close(self):
        if getattr(self, "h", None):
            self.lib.himgcu_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, allow=()):
        if rc != _native.OK and rc not in allow:
            raise HimgError(rc, self.lib.himgcu_last_error(self.h).decode())
        return rc

    def set_stream(self, stream):
        """stream: raw cudaStream_t handle (int; 0 = CUDA's legacy default stream) or a
        torch.cuda.Stream; None goes back to the context's own non-blocking stream."""
        self._bound = None
        if stream is None:
            self._explicit_stream = False
            self._check(self.lib.himgcu_reset_stream(self.h))
            return
        self._explicit_stream = True
        handle = getattr(stream, "cuda_stream", stream)
        self._check(self.lib.himgcu_set_stream(self.h, C.c_void_p(int(handle))))

    def _bind(self, *tensors, rows_ok=False):
        """Called by every method that takes or returns torch tensors.  Checks that they are contiguous
        uint8 / integer tensors on this context's device and -- unless the user chose a stream with
        set_stream() -- runs the call on torch's CURRENT stream of that device, the stream the tensors were
        produced on and will be consumed on (the context's own stream is not ordered against it)."""
        import torch

        for x in tensors:
            if x is None:
                continue
            if not x.is_cuda or (x.device.index or 0) != self.device:
                raise ValueError(f"tensor on {x.device}, the context is on cuda:{self.device}")
            if not (x.is_contiguous() or (rows_ok and x.dim() >= 2 and x[0].is_contiguous())):
                raise ValueError("tensors must be contiguous")
        if not self._explicit_stream:
            handle = torch.cuda.current_stream(self.device).cuda_stream
            if handle != self._bound:
                self._check(self.lib.himgcu_set_stream(self.h, C.c_void_p(int(handle))))
                self._bound = handle

    def encode_status(self):
        """Synchronises and raises if an image of an earlier encode_batch could not be encoded."""
        self._check(self.lib.himgcu_encode_status(self.h))

    def synchronize(self):
        self._check(self.lib.himgcu_synchronize(self.h))

    # ---- single image, host buffers -------------------------------------------------------
    def encode(self, img: np.ndarray, quality=50, use_ycbcr=True, pixel_stride=None, w=None, h=None, nch=None) -> bytes:
        img = np.ascontiguousarray(img, np.uint8)
        if w is None:
            h, w, nch = img.shape
        ps = pixel_stride or nch
        out = np.empty(encode_bound(w, h, nch), np.uint8)
        n = C.c_size_t()
        self._check(self.lib.himgcu_encode(self.h, _ptr(img), w, h, ps, nch, quality, int(use_ycbcr), _ptr(out), out.size,
                                           C.byref(n)))
        return out[: n.value].tobytes()

    def _decode_single(self, data: bytes, shape, fn, *args):
        """Body of decode, decode_scaled, decode_region and decode_region_scaled: probes the header, allocates
        shape(w, h, nch) and calls the C entry point fn with args after the stream.  None where the stream is rejected."""
        buf = np.frombuffer(data, np.uint8)
        w, h, n = C.c_int(), C.c_int(), C.c_int()
        if self.lib.himgcu_decode_info(_ptr(buf), buf.size, C.byref(w), C.byref(h), C.byref(n)) != _native.OK:
            return None
        if w.value < 1 or h.value < 1 or n.value < 1:
            return None
        out = np.empty(shape(w.value, h.value, n.value), np.uint8)
        rc = self._check(fn(self.h, _ptr(buf), buf.size, *args, _ptr(out), out.size, C.byref(w), C.byref(h), C.byref(n)),
                         allow=(_native.REJECT,))
        return None if rc == _native.REJECT else out

    def decode(self, data: bytes, flags=STRICT):
        """Returns the decoded [h][w][nch] array, or None where the reference decoder returns false."""
        return self._decode_single(data, lambda w, h, n: (h, w, n), self.lib.himgcu_decode, flags)

    def decode_scaled(self, data: bytes, factor: int, flags=STRICT):
        """The image at 1/factor size (factor 1, 2, 4 or 8): the [ceil(h/f)][ceil(w/f)][nch] array of rounded box
        averages of decode(data) over f x f windows (clipped at the right and bottom edges), or None where the stream
        is rejected.  Raises HimgError (ERR_ARG) for another factor."""
        f = max(int(factor), 1)
        return self._decode_single(data, lambda w, h, n: (-(-h // f), -(-w // f), n), self.lib.himgcu_decode_scaled, flags,
                                   factor)

    def decode_region(self, data: bytes, x: int, y: int, w: int, h: int, flags=STRICT):
        """Rectangle [x, x+w) x [y, y+h) of the image: the [h][w][nch] array equal to decode(data)[y:y+h, x:x+w],
        or None where the stream is rejected.  Raises HimgError for an empty rectangle or one outside the image."""
        return self._decode_single(data, lambda W, H, n: (max(h, 1), max(w, 1), n), self.lib.himgcu_decode_region, flags, x, y,
                                   w, h)

    def decode_region_scaled(self, data: bytes, factor: int, x: int, y: int, w: int, h: int, flags=STRICT):
        """Rectangle [x, x+w) x [y, y+h) of the image at 1/factor size (factor 1, 2, 4 or 8): the [h][w][nch] array
        equal to decode_scaled(data, factor)[y:y+h, x:x+w], or None where the stream is rejected.  Only the block rows
        of the source rectangle are entropy-decoded, so the status is that of decode_region on it.  Raises HimgError
        (ERR_ARG) for another factor, an empty rectangle or one outside the scaled image."""
        return self._decode_single(data, lambda W, H, n: (max(h, 1), max(w, 1), n), self.lib.himgcu_decode_region_scaled, flags,
                                   factor, x, y, w, h)

    # ---- batch, device tensors --------------------------------------------------------------
    def encode_batch(self, pixels, quality=50, use_ycbcr=True, out=None, sizes=None):
        """pixels: CUDA uint8 tensor [n][h][w][nch].  Returns (out [n][stride] u8, sizes [n] i32)."""
        import torch

        n, h, w, nch = pixels.shape
        stride = (encode_bound(w, h, nch) + 255) & ~255
        if pixels.dtype != torch.uint8:
            raise ValueError("pixels must be uint8")
        self._bind(pixels, out, sizes)
        if out is None:
            out = torch.empty((n, stride), dtype=torch.uint8, device=pixels.device)
        if sizes is None:
            sizes = torch.empty((n,), dtype=torch.int32, device=pixels.device)
        self._check(self.lib.himgcu_encode_batch(self.h, _ptr(pixels), n, w, h, nch, quality, int(use_ycbcr), _ptr(out),
                                                 out.stride(0), _ptr(sizes)))
        return out, sizes

    def _decode_batch(self, fn, himg, offsets, sizes, w, h, nch, factor, out, status, *args):
        """Body of decode_batch and decode_batch_scaled: fn is the C entry point, args its arguments after nch."""
        import torch

        n = offsets.numel()
        self._bind(himg, offsets, sizes, out, status)
        if out is None:
            f = max(int(factor), 1)
            out = torch.empty((n, -(-h // f), -(-w // f), nch), dtype=torch.uint8, device=himg.device)
        if status is None:
            status = torch.empty((n,), dtype=torch.int32, device=himg.device)
        self._check(fn(self.h, _ptr(himg), _ptr(offsets), _ptr(sizes), n, w, h, nch, *args, _ptr(out), _ptr(status)))
        return out, status

    def decode_batch(self, himg, offsets, sizes, w, h, nch, flags=STRICT, out=None, status=None):
        """himg: CUDA uint8 buffer; offsets int64 [n], sizes int32 [n] (device).  Returns (pixels, status)."""
        return self._decode_batch(self.lib.himgcu_decode_batch, himg, offsets, sizes, w, h, nch, 1, out, status, flags)

    def _decode_batch_region(self, fn, himg, offsets, sizes, dims, origins, crop_w, crop_h, nch, out, status, *args):
        """Body of the decode_batch_region calls: fn is the C entry point, args its arguments between n and the origins
        (dims is None for a uniform batch)."""
        import torch

        n = offsets.numel()
        for name, t in (("dims", dims), ("origins", origins)):
            if t is not None and (t.dtype != torch.int32 or t.numel() != 2 * n):
                raise ValueError(name + " must be an int32 tensor [n][2]")
        self._bind(himg, offsets, sizes, dims, origins, out, status)
        if out is None:
            out = torch.empty((n, crop_h, crop_w, nch), dtype=torch.uint8, device=himg.device)
        if status is None:
            status = torch.empty((n,), dtype=torch.int32, device=himg.device)
        self._check(fn(self.h, _ptr(himg), _ptr(offsets), _ptr(sizes), n, *args, _ptr(origins), crop_w, crop_h, _ptr(out),
                       _ptr(status)))
        return out, status

    def decode_batch_region(self, himg, offsets, sizes, w, h, nch, origins, crop_w, crop_h, flags=STRICT, out=None,
                            status=None):
        """decode_batch of a crop_w x crop_h rectangle per image: origins is a CUDA int32 [n][2] tensor of (x, y).
        Returns (pixels [n][crop_h][crop_w][nch], status); status[i] is ERR_ARG where the origin puts the
        rectangle outside the image (that image's pixels are not written)."""
        return self._decode_batch_region(self.lib.himgcu_decode_batch_region, himg, offsets, sizes, None, origins, crop_w, crop_h,
                                         nch, out, status, w, h, nch, flags)

    def decode_batch_region_mixed(self, himg, offsets, sizes, dims, nch, origins, crop_w, crop_h, max_w, max_h, flags=STRICT,
                                  out=None, status=None):
        """decode_batch_region of streams with their own sizes: dims is a CUDA int32 [n][2] tensor of (width, height),
        each at most max_w x max_h, and origins one of (x, y).  Returns (pixels [n][crop_h][crop_w][nch], status);
        status[i] is REJECT where the stream is rejected or its shape is not dims[i] x nch, and ERR_ARG where dims[i]
        is < 1 or exceeds the bounds or the origin puts the rectangle outside the image (those pixels are not written)."""
        return self._decode_batch_region(self.lib.himgcu_decode_batch_region_mixed, himg, offsets, sizes, dims, origins, crop_w,
                                         crop_h, nch, out, status, _ptr(dims), max_w, max_h, nch, flags)

    def decode_batch_region_scaled(self, himg, offsets, sizes, w, h, nch, factor, origins, crop_w, crop_h, flags=STRICT, out=None,
                                   status=None):
        """decode_batch_region of the images at 1/factor size (factor 1, 2, 4 or 8, see decode_region_scaled): origins
        and crop_w x crop_h are in the scaled images' coordinates, and crop_w x crop_h must fit ceil(w/f) x ceil(h/f).
        Returns (pixels [n][crop_h][crop_w][nch], status) with the statuses of decode_batch_region."""
        return self._decode_batch_region(self.lib.himgcu_decode_batch_region_scaled, himg, offsets, sizes, None, origins, crop_w,
                                         crop_h, nch, out, status, w, h, nch, flags, factor)

    def decode_batch_region_mixed_scaled(self, himg, offsets, sizes, dims, nch, factor, origins, crop_w, crop_h, max_w, max_h,
                                         flags=STRICT, out=None, status=None):
        """decode_batch_region_mixed of the images at 1/factor size: origins are checked against each image's scaled
        shape, and crop_w x crop_h against ceil(max_w/f) x ceil(max_h/f).  Returns (pixels [n][crop_h][crop_w][nch],
        status) with the statuses of decode_batch_region_mixed."""
        return self._decode_batch_region(self.lib.himgcu_decode_batch_region_mixed_scaled, himg, offsets, sizes, dims, origins,
                                         crop_w, crop_h, nch, out, status, _ptr(dims), max_w, max_h, nch, flags, factor)

    def _decode_batch_mixed(self, fn, himg, offsets, sizes, dims, nch, max_w, max_h, factor, out, pixel_offsets, status, *args):
        """Body of decode_batch_mixed (factor None) and decode_batch_mixed_scaled: fn is the C entry point, args its
        arguments after nch."""
        import torch

        n = offsets.numel()
        if dims.dtype != torch.int32 or dims.numel() != 2 * n:
            raise ValueError("dims must be an int32 tensor [n][2]")
        if pixel_offsets is not None and (pixel_offsets.dtype != torch.int64 or pixel_offsets.numel() != n):
            raise ValueError("pixel_offsets must be an int64 tensor [n]")
        self._bind(himg, offsets, sizes, dims, out, pixel_offsets, status)
        if pixel_offsets is None or out is None:  # (an image with dims out of bounds gets an empty span)
            wh = dims.reshape(n, 2).to(torch.int64)
            ok = (wh >= 1).all(dim=1) & (wh[:, 0] <= max_w) & (wh[:, 1] <= max_h)
            if factor is not None:
                f = max(int(factor), 1)
                wh = torch.div(wh + (f - 1), f, rounding_mode="floor")
            spans = torch.where(ok, wh[:, 0] * wh[:, 1] * nch, 0)
        if pixel_offsets is None:
            pixel_offsets = torch.cumsum(spans, 0) - spans
        if out is None:
            total = int(spans.sum()) if n else 0
            out = torch.empty((max(total, 1),), dtype=torch.uint8, device=himg.device)
        if status is None:
            status = torch.empty((n,), dtype=torch.int32, device=himg.device)
        self._check(fn(self.h, _ptr(himg), _ptr(offsets), _ptr(sizes), n, _ptr(dims), max_w, max_h, nch, *args, _ptr(pixel_offsets),
                       _ptr(out), _ptr(status)))
        return out, pixel_offsets, status

    def decode_batch_mixed(self, himg, offsets, sizes, dims, nch, max_w, max_h, flags=STRICT, out=None, pixel_offsets=None,
                           status=None):
        """decode_batch of streams with their own sizes: dims is a CUDA int32 [n][2] tensor of (w_i, h_i), each at most
        max_w x max_h.  Image i is written as [h_i][w_i][nch] at byte pixel_offsets[i] (int64 [n]) of the flat uint8
        buffer out.  When pixel_offsets is None they are the exclusive prefix sum of w_i * h_i * nch (0 for dims out of
        bounds), computed on the device; when out is None it is allocated for the spans, which reads their total back
        to the host (one synchronisation).  Returns (out, pixel_offsets, status); status[i] is REJECT where the stream is rejected or its
        shape is not dims[i] x nch, and ERR_ARG where dims[i] is < 1 or exceeds the bounds (nothing of it is written)."""
        return self._decode_batch_mixed(self.lib.himgcu_decode_batch_mixed, himg, offsets, sizes, dims, nch, max_w, max_h, None, out,
                                        pixel_offsets, status, flags)

    def decode_batch_scaled(self, himg, offsets, sizes, w, h, nch, factor, flags=STRICT, out=None, status=None):
        """decode_batch at 1/factor size (factor 1, 2, 4 or 8, see decode_scaled).  Returns (pixels
        [n][ceil(h/f)][ceil(w/f)][nch], status)."""
        return self._decode_batch(self.lib.himgcu_decode_batch_scaled, himg, offsets, sizes, w, h, nch, factor, out, status, flags,
                                  factor)

    def decode_batch_mixed_scaled(self, himg, offsets, sizes, dims, nch, max_w, max_h, factor, flags=STRICT, out=None,
                                  pixel_offsets=None, status=None):
        """decode_batch_mixed at 1/factor size (factor 1, 2, 4 or 8, see decode_scaled): image i is written as
        [ceil(h_i/f)][ceil(w_i/f)][nch] at byte pixel_offsets[i] of the flat uint8 buffer out.  When pixel_offsets is
        None they are the exclusive prefix sum of those spans (0 for dims out of bounds), computed on the device; when
        out is None it is allocated for the spans (one synchronisation).  Returns (out, pixel_offsets, status), with
        the statuses of decode_batch_mixed."""
        return self._decode_batch_mixed(self.lib.himgcu_decode_batch_mixed_scaled, himg, offsets, sizes, dims, nch, max_w, max_h,
                                        factor, out, pixel_offsets, status, flags, factor)

    def encode_batch_mixed(self, pixels, offsets, dims, nch, max_w, max_h, quality=50, use_ycbcr=True, out=None, sizes=None):
        """encode_batch of images with their own sizes: pixels is a flat CUDA uint8 buffer holding image i as
        [h_i][w_i][nch] at byte offsets[i] (int64 [n]), dims a CUDA int32 [n][2] tensor of (w_i, h_i), each at most
        max_w x max_h.  Returns (out [n][stride] u8, sizes [n] i32); image i's stream is what encode_batch gives for it
        alone.  sizes[i] is 0 where dims[i] is < 1 or exceeds the bounds (encode_status then raises ERR_ARG) or the
        stream does not fit the stride (ERR_CAPACITY); nothing is written to such an image's row of out."""
        import torch

        n = offsets.numel()
        if pixels.dtype != torch.uint8:
            raise ValueError("pixels must be uint8")
        if offsets.dtype != torch.int64:
            raise ValueError("offsets must be an int64 tensor [n]")
        if dims.dtype != torch.int32 or dims.numel() != 2 * n:
            raise ValueError("dims must be an int32 tensor [n][2]")
        self._bind(pixels, offsets, dims, out, sizes)
        stride = (encode_bound(max_w, max_h, nch) + 255) & ~255
        if out is None:
            out = torch.empty((n, stride), dtype=torch.uint8, device=pixels.device)
        if sizes is None:
            sizes = torch.empty((n,), dtype=torch.int32, device=pixels.device)
        self._check(self.lib.himgcu_encode_batch_mixed(self.h, _ptr(pixels), _ptr(offsets), _ptr(dims), n, max_w, max_h, nch,
                                                       quality, int(use_ycbcr), _ptr(out), out.stride(0),
                                                       _ptr(sizes)))
        return out, sizes

    # ---- batch, host buffers (numpy arrays or pinned CPU torch tensors) -------------------------
    def encode_batch_host(self, pixels, quality=50, use_ycbcr=True, out=None, offsets=None, sizes=None):
        """pixels: host uint8 [n][h][w][nch].  Returns (out u8 buffer, offsets u64 [n+1], sizes u32 [n])."""
        n, h, w, nch = pixels.shape
        if out is None:
            out = np.empty(n * encode_bound(w, h, nch), np.uint8)
        if offsets is None:
            offsets = np.empty(n + 1, np.uint64)
        if sizes is None:
            sizes = np.empty(n, np.uint32)
        cap = out.size if isinstance(out, np.ndarray) else out.numel()
        self._check(self.lib.himgcu_encode_batch_host(self.h, _ptr(pixels), n, w, h, nch, quality, int(use_ycbcr),
                                                      _ptr(out), cap, _ptr(offsets), _ptr(sizes)))
        return out, offsets, sizes

    def decode_batch_host(self, himg, offsets, sizes, w, h, nch, flags=STRICT, out=None, status=None):
        n = (offsets.size if isinstance(offsets, np.ndarray) else offsets.numel()) - 1
        if out is None:
            out = np.empty((n, h, w, nch), np.uint8)
        if status is None:
            status = np.empty(n, np.int32)
        self._check(self.lib.himgcu_decode_batch_host(self.h, _ptr(himg), _ptr(offsets), _ptr(sizes), n, w, h, nch, flags,
                                                      _ptr(out), _ptr(status)))
        return out, status

    # ---- stages (device tensors) ---------------------------------------------------------------
    def stage_lowres(self, pixels, use_ycbcr=True, nch=None):
        import torch

        n, h, w, ps = pixels.shape
        self._bind(pixels)
        nch = nch or ps
        rows, cols = (h + 7) >> 3, (w + 7) >> 3
        L = torch.empty((n, nch, rows, cols), dtype=torch.uint8, device=pixels.device)
        self._check(self.lib.himgcu_stage_lowres(self.h, _ptr(pixels), n, w, h, ps, nch, int(use_ycbcr), _ptr(L)))
        return L

    def stage_lres_encode(self, L, w, h, quality):
        import torch

        n, nch = L.shape[0], L.shape[1]
        self._bind(L)
        stride = int(self.lib.himgcu_lres_stride(w, h, nch))
        size = int(self.lib.himgcu_lres_size(w, h, nch))
        out = torch.zeros((n, stride), dtype=torch.uint8, device=L.device)
        self._check(self.lib.himgcu_stage_lres_encode(self.h, _ptr(L), n, w, h, nch, quality, _ptr(out)))
        return out, size

    def stage_forward(self, pixels, L, quality=50, use_ycbcr=True, nch=None):
        import torch

        n, h, w, ps = pixels.shape
        self._bind(pixels, L)
        nch = nch or ps
        rows, cols = (h + 7) >> 3, (w + 7) >> 3
        planes = torch.empty((n, rows * cols * 64 * nch), dtype=torch.uint8, device=pixels.device)
        self._check(self.lib.himgcu_stage_forward(self.h, _ptr(pixels), _ptr(L), n, w, h, ps, nch, quality, int(use_ycbcr),
                                                  _ptr(planes)))
        return planes

    def stage_huff_compress(self, data, block_size=0):
        """data: CUDA uint8 [n][in_size].  Returns (out [n][stride], sizes [n])."""
        import torch

        n, in_size = data.shape
        self._bind(data, rows_ok=True)  # (the row stride travels with the call)
        stride = (2 * in_size + 4096 + 255) & ~255
        out = torch.zeros((n, stride), dtype=torch.uint8, device=data.device)
        sizes = torch.zeros((n,), dtype=torch.int32, device=data.device)
        self._check(self.lib.himgcu_stage_huff_compress(self.h, _ptr(data), data.stride(0), n, in_size, block_size,
                                                        _ptr(out), stride, _ptr(sizes)))
        return out, sizes

    def stage_huff_uncompress(self, packed, sizes, out_size, block_size=0, flags=STRICT):
        import torch

        n = packed.shape[0]
        self._bind(packed, sizes, rows_ok=True)
        stride = (out_size + 63) & ~63
        out = torch.zeros((n, stride), dtype=torch.uint8, device=packed.device)
        status = torch.zeros((n,), dtype=torch.int32, device=packed.device)
        self._check(self.lib.himgcu_stage_huff_uncompress(self.h, _ptr(packed), packed.stride(0), _ptr(sizes), n, out_size,
                                                          block_size, flags, _ptr(out), stride, _ptr(status)))
        return out[:, :out_size], status

    def stage_lres_decode(self, lres, w, h, nch, unmap):
        import torch

        n = lres.shape[0]
        self._bind(lres, rows_ok=True)
        rows, cols = (h + 7) >> 3, (w + 7) >> 3
        un = np.ascontiguousarray(unmap, np.int16)
        R = torch.zeros((n, nch, rows, cols), dtype=torch.uint8, device=lres.device)
        self._check(self.lib.himgcu_stage_lres_decode(self.h, _ptr(lres), lres.stride(0), n, w, h, nch, _ptr(un), _ptr(R)))
        return R

    def stage_inverse(self, planes, R, w, h, nch, use_ycbcr, shift_luma, shift_chroma, unmap):
        import torch

        n = planes.shape[0]
        self._bind(planes, R)
        sl = np.ascontiguousarray(shift_luma, np.uint8)
        sc = np.ascontiguousarray(shift_chroma, np.uint8)
        un = np.ascontiguousarray(unmap, np.int16)
        out = torch.zeros((n, h, w, nch), dtype=torch.uint8, device=planes.device)
        self._check(self.lib.himgcu_stage_inverse(self.h, _ptr(planes), _ptr(R), n, w, h, nch, int(use_ycbcr), _ptr(sl),
                                                  _ptr(sc), _ptr(un), _ptr(out)))
        return out

    # ---- profiling -----------------------------------------------------------------------------
    def profile(self, on=True):
        self._check(self.lib.himgcu_profile_enable(self.h, int(on)))

    def profile_reset(self):
        self._check(self.lib.himgcu_profile_reset(self.h))

    def profile_results(self) -> dict:
        out = {}
        for i in range(self.lib.himgcu_profile_count(self.h)):
            name, ms, cnt = C.c_char_p(), C.c_double(), C.c_int()
            self.lib.himgcu_profile_get(self.h, i, C.byref(name), C.byref(ms), C.byref(cnt))
            out[name.value.decode()] = (ms.value, cnt.value)
        return out

    def set_option(self, name: str, value: int):
        self._check(self.lib.himgcu_set_option(self.h, name.encode(), int(value)))

    def launch_count(self) -> int:
        return int(self.lib.himgcu_launch_count(self.h))


class Encoder:
    """Mirror of himg::Encoder (src/lib/encoder.h:20-64): Encode(...) -> bool, packed_data()."""

    def __init__(self, ctx: Context | None = None):
        self._ctx = ctx or Context(0)
        self._packed = b""

    def Encode(self, data, width, height, pixel_stride, num_channels, quality, use_ycbcr) -> bool:
        self._packed = self._ctx.encode(np.frombuffer(data, np.uint8) if not isinstance(data, np.ndarray) else data,
                                        quality, use_ycbcr, pixel_stride, width, height, num_channels)
        return True

    def packed_data(self) -> bytes:
        return self._packed

    def packed_size(self) -> int:
        return len(self._packed)


class Decoder:
    """Mirror of himg::Decoder (src/lib/decoder.h:22-67).  max_threads is accepted and ignored."""

    def __init__(self, max_threads: int = 0, ctx: Context | None = None, flags=STRICT):
        self._ctx = ctx or Context(0)
        self._flags = flags
        self._img = None

    def Decode(self, packed_data, packed_size=None) -> bool:
        data = bytes(packed_data[:packed_size] if packed_size is not None else packed_data)
        self._img = self._ctx.decode(data, self._flags)
        return self._img is not None

    def unpacked_data(self):
        return self._img

    def unpacked_size(self) -> int:
        return 0 if self._img is None else self._img.size

    def width(self) -> int:
        return 0 if self._img is None else self._img.shape[1]

    def height(self) -> int:
        return 0 if self._img is None else self._img.shape[0]

    def num_channels(self) -> int:
        return 0 if self._img is None else self._img.shape[2]
