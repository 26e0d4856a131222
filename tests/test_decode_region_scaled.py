"""Scaled region decode (himgcu_decode_region_scaled, himgcu_decode_batch_region_scaled,
himgcu_decode_batch_region_mixed_scaled): a rectangle of the image at 1/f size, in the scaled image's coordinates.

The reference is the oracle's whole decode, box-averaged in numpy (the contract of the scaled calls) and cropped.  The
status of a call is that of himgcu_decode_region on the source rectangle (f x, f y, min(f rw, W - f x), min(f rh, H - f y)),
so a stream whose corruption lies below the rectangle may decode.  Output buffers are filled with a sentinel and are
longer than the batch's output, so a write outside an image's own rectangle is seen."""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")

OK, REJECT, ERR_ARG, ERR_CAPACITY = 0, 1, 2, 4
FILL = 0x5A
FACTORS = (2, 4, 8)
ODD = [(1, 1), (17, 3), (37, 21), (300, 5), (2056, 16), (1920, 1080), (3840, 2160)]
gpu = pytest.mark.gpu


def cdiv(a, f):
    return -(-a // f)


# ---------------------------------------------------------------------------------------------
# CPU: the bounds the host sizes its buffers and grids with
# ---------------------------------------------------------------------------------------------
def region_rows(rh, f, rows):
    """Compact block rows per image (api.cu region_rows)."""
    return min((f * rh + 15 - f) // 8, rows)


def region_span_pairs(rw, cols):
    """Block pairs a slot of the lane-pair region kernels stages (xform_region.cuh), for a source width rw."""
    kb = (rw + 14) // 8
    return min(8 * ((kb + 30) // 16), cols // 2)


@pytest.mark.parametrize("f", [1, 2, 4, 8])
def test_rows_touched_never_exceed_the_bound(f):
    for H in [1, 3, 7, 8, 9, 15, 16, 17, 21, 63, 64, 65, 100, 129, 200, 257]:
        rows, sh = cdiv(H, 8), cdiv(H, f)
        for rh in range(1, min(64, sh) + 1):
            kr = region_rows(rh, f, rows)
            y = np.arange(0, sh - rh + 1)
            r0 = (f * y) >> 3
            r1 = (np.minimum(f * (y + rh), H) - 1) >> 3
            touched = r1 - r0 + 1
            assert touched.max() <= kr, (f, H, rh)
            if H >= f * rh + 8:  # (a tall image reaches the bound at some y phase)
                assert touched.max() == kr, (f, H, rh)
    assert all(region_rows(rh, 1, 1 << 20) == (rh + 14) // 8 for rh in range(1, 200))
    assert all(region_rows(rh, 8, 1 << 20) == rh for rh in range(1, 200))


@pytest.mark.parametrize("f", [2, 4, 8])
def test_columns_touched_fit_the_lane_pair_span(f):
    """On the shapes of the lane-pair kernel (w % 16 == 0) every block column a rectangle reads lies inside the span
    staged from the 16-block boundary at or below its first column."""
    for W in [16, 32, 48, 128, 256, 400, 1024, 1920]:
        cols, sw = W // 8, W // f
        for rw in list(range(1, min(64, sw) + 1)) + [sw]:
            span = region_span_pairs(f * rw, cols)
            x = np.arange(0, sw - rw + 1)
            u0 = ((f * x) >> 3) & ~15
            ur = (f * (x + rw) - 1) >> 3
            assert (ur < u0 + 2 * span).all(), (f, W, rw)
            assert (ur < cols).all()


# ---------------------------------------------------------------------------------------------
# GPU helpers
# ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ctx():
    import himg_b200

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    c = himg_b200.Context(0)
    c.set_stream(torch.cuda.current_stream().cuda_stream)
    yield c
    c.close()


@pytest.fixture(scope="module")
def generic():
    import himg_b200

    c = himg_b200.Context(0)
    c.set_stream(torch.cuda.current_stream().cuda_stream)
    c.set_option("force_generic", 1)
    yield c
    c.close()


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def assert_same(got, want, what):
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, f"{what}: shape {got.shape} vs {want.shape}"
    idx = np.flatnonzero(got.reshape(-1) != want.reshape(-1))
    assert idx.size == 0, f"{what}: {idx.size} diffs, first at {int(idx[0])}"


def box(d, f):
    """Rounded box averages of d [H][W][C] over f x f windows, clipped at the right and bottom edges (copied from
    test_decode_scaled.py)."""
    if d is None or f == 1:
        return d
    H, W, nch = d.shape
    oh, ow = cdiv(H, f), cdiv(W, f)
    p = np.zeros((oh * f, ow * f, nch), np.int64)
    p[:H, :W] = d
    s = p.reshape(oh, f, ow, f, nch).sum(axis=(1, 3))
    n = (np.minimum(f, H - f * np.arange(oh))[:, None] * np.minimum(f, W - f * np.arange(ow))[None, :])[..., None]
    return ((s + n // 2) // n).astype(np.uint8)


def pack(streams):
    offs = np.cumsum([0] + [(len(s) + 15) & ~15 for s in streams])
    buf = np.zeros(offs[-1] + 64, np.uint8)
    for o, s in zip(offs, streams):
        buf[o: o + len(s)] = np.frombuffer(s, np.uint8)
    return dev(buf), dev(offs[:-1].astype(np.int64)), dev(np.array([len(s) for s in streams], np.int32))


_streams = {}


def stream(port, w, h, nch, q=50, ycbcr=True, seed=None):
    """(stream, {flags: box-averaged whole decode per factor}) of the oracle, cached across tests."""
    key = (w, h, nch, q, ycbcr, seed)
    if key not in _streams:
        s = port.encode(port.synth(w, h, nch, seed if seed is not None else (w * 7 + h) % 97, 6), q, ycbcr)
        full = (port.decode(s), port.decode(s, strict=False))
        _streams[key] = (s, {(fl, f): box(full[fl], f) for fl in (0, 1) for f in (1, 2, 4, 8)})
    return _streams[key]


def run_batch(c, streams, w, h, nch, f, origins, rw, rh, flags=0, mixed_dims=None, max_wh=None, spare=5):
    """One batch call into a sentinel-filled buffer `spare` images longer than the batch: (images, status, whether the
    bytes past the batch kept the sentinel)."""
    n = len(streams)
    out = torch.full(((n + spare) * rh * rw * nch,), FILL, dtype=torch.uint8, device="cuda")
    view = out[: n * rh * rw * nch].view(n, rh, rw, nch)
    himg, offs, sizes = pack(streams)
    org = dev(np.asarray(origins, np.int32).reshape(-1, 2))
    if mixed_dims is None:
        _, status = c.decode_batch_region_scaled(himg, offs, sizes, w, h, nch, f, org, rw, rh, flags, out=view)
    else:
        _, status = c.decode_batch_region_mixed_scaled(himg, offs, sizes, dev(np.asarray(mixed_dims, np.int32).reshape(-1, 2)),
                                                       nch, f, org, rw, rh, *max_wh, flags, out=view)
    buf = out.cpu().numpy()
    return buf[: view.numel()].reshape(n, rh, rw, nch), status.cpu().numpy(), bool((buf[view.numel():] == FILL).all())


def kernels_of(c, fn):
    c.profile(True)
    c.profile_reset()
    try:
        fn()
        c.synchronize()
        return set(c.profile_results())
    finally:
        c.profile(False)


def rects(sw, sh, f):
    """Rectangles of a sw x sh scaled image: 1 x 1 at both corners, every x and y phase modulo 8 / f, rectangles with the
    clipped edge windows, one inside one block row, and the whole image."""
    out = [(0, 0, 1, 1), (sw - 1, sh - 1, 1, 1), (0, 0, sw, sh)]
    p = 8 // f
    for px in range(p):
        for py in range(p):
            x, y = min(px + p, sw - 1), min(py, sh - 1)
            out.append((x, y, min(sw - x, 5 + px), min(sh - y, 3 + py)))
    out.append((max(0, sw - 7), max(0, sh - 4), min(sw, 7), min(sh, 4)))  # the right and bottom edges
    out.append((min(1, sw - 1), 0, max(1, sw - 2), min(sh, max(1, p - 1))))  # inside the first block row
    return list(dict.fromkeys(out))


def check_rects(c, s, want, w, h, nch, f, flags, what, single=True):
    sw, sh = cdiv(w, f), cdiv(h, f)
    for (x, y, rw, rh) in rects(sw, sh, f):
        imgs, status, untouched = run_batch(c, [s, s], w, h, nch, f, [(x, y), (x, y)], rw, rh, flags)
        tag = f"{what} rect {(x, y, rw, rh)}"
        assert untouched, tag + ": written past the batch"
        if want is None:  # (the strict decoder refuses the unframed FRES chunk of an image of one block row)
            assert list(status) == [REJECT, REJECT], tag
            assert not single or c.decode_region_scaled(s, f, x, y, rw, rh, flags) is None, tag
            continue
        assert list(status) == [OK, OK], tag
        for k in range(2):
            assert_same(imgs[k], want[y: y + rh, x: x + rw], tag + f" image {k}")
        if single:
            assert_same(c.decode_region_scaled(s, f, x, y, rw, rh, flags), want[y: y + rh, x: x + rw], tag + " single")


# ---------------------------------------------------------------------------------------------
# against the oracle
# ---------------------------------------------------------------------------------------------
CHANNELS = [(1, True), (2, True), (3, True), (3, False), (4, True), (5, False), (6, True)]


@gpu
@pytest.mark.parametrize("nch, ycbcr", CHANNELS)
def test_odd_shapes_match_oracle(ctx, port, nch, ycbcr):
    for (w, h) in ODD:
        s, wants = stream(port, w, h, nch, 50, ycbcr)
        for f in FACTORS:
            for flags in (0, 1):
                check_rects(ctx, s, wants[(flags, f)], w, h, nch, f, flags, f"{w}x{h}x{nch} ycbcr {ycbcr} f {f} flags {flags}",
                            single=max(w, h) < 3000)
        _streams.pop((w, h, nch, 50, ycbcr, None))  # (the 4K decodes are large)


@gpu
@pytest.mark.parametrize("q", [0, 100])
def test_qualities_and_generic(ctx, generic, port, q):
    """q0 (strict-rejected whole, lenient decoded) and q100 through both inverse kernels."""
    for (w, h, nch) in [(1920, 1080, 3), (1024, 64, 1), (300, 77, 3)]:
        s, wants = stream(port, w, h, nch, q)
        for f in FACTORS:
            sw, sh = cdiv(w, f), cdiv(h, f)
            rw, rh = min(sw, 29), min(sh, 13)
            origins = [(0, 0), (sw - rw, sh - rh), (3 % (sw - rw + 1), 5 % (sh - rh + 1))]
            for flags in (0, 1):
                want = wants[(flags, f)]
                for c in (ctx, generic):
                    imgs, status, untouched = run_batch(c, [s] * 3, w, h, nch, f, origins, rw, rh, flags)
                    assert untouched
                    if want is None:
                        assert list(status) == [REJECT] * 3, (w, h, nch, f, flags)
                        continue
                    assert list(status) == [OK] * 3, (w, h, nch, f, flags)
                    for k, (x, y) in enumerate(origins):
                        assert_same(imgs[k], want[y: y + rh, x: x + rw], f"q{q} {w}x{h}x{nch} f {f} flags {flags} image {k}")


# ---------------------------------------------------------------------------------------------
# the lane-pair kernel against the generic one, and which kernel runs
# ---------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("w, h, nch", [(1920, 1080, 3), (3840, 2160, 3), (1024, 1024, 1)])
def test_lane_pair_equals_generic(ctx, generic, port, w, h, nch):
    s = stream(port, w, h, nch, 70)[0]
    for f in FACTORS:
        sw, sh = w // f, h // f
        # rw * nch odd: the output rows of the 16 rows of a rectangle start at every alignment modulo 16, and the origins
        # take every x phase modulo 16 output pixels
        for rw, rh in ((min(37, sw), min(16, sh)), (min(sw, 225), min(sh, 19)), (sw, sh)):
            origins = [((7 * k) % (sw - rw + 1), (5 * k) % (sh - rh + 1)) for k in range(16)]
            n = len(origins)
            himg, offs, sizes = pack([s] * n)
            org = dev(np.asarray(origins, np.int32))
            k = kernels_of(ctx, lambda: ctx.decode_batch_region_scaled(himg, offs, sizes, w, h, nch, f, org, rw, rh))
            assert "k_inverse_region4_scaled" in k and "k_inverse_region_scaled" not in k, k
            k = kernels_of(generic, lambda: generic.decode_batch_region_scaled(himg, offs, sizes, w, h, nch, f, org, rw, rh))
            assert "k_inverse_region_scaled" in k and "k_inverse_region4_scaled" not in k, k
            a, sa = run_batch(ctx, [s] * n, w, h, nch, f, origins, rw, rh)[:2]
            b, sb = run_batch(generic, [s] * n, w, h, nch, f, origins, rw, rh)[:2]
            assert list(sa) == list(sb) == [OK] * n
            assert_same(a, b, f"{w}x{h}x{nch} f {f} {rw}x{rh}: lane-pair vs generic")
    ctx.set_option("xform_variant", 1)
    try:
        k = kernels_of(ctx, lambda: ctx.decode_batch_region_scaled(himg, offs, sizes, w, h, nch, 2, org, 8, 8))
        assert "k_inverse_region_scaled" in k and "k_inverse_region4_scaled" not in k, k
    finally:
        ctx.set_option("xform_variant", 0)


# ---------------------------------------------------------------------------------------------
# equalities between calls
# ---------------------------------------------------------------------------------------------
@gpu
def test_factor_one_is_the_region_call(ctx, port):
    garbage = b"RIFF" + b"\1" * 40
    for (w, h, nch) in [(1920, 1080, 3), (1024, 1024, 1), (37, 21, 5), (300, 77, 3)]:
        s = stream(port, w, h, nch)[0]
        rw, rh = min(w, 224), min(h, 100)
        origins = [(0, 0), (w - rw, h - rh), (3 % (w - rw + 1), 11 % (h - rh + 1))]
        streams = [s, garbage, s]
        himg, offs, sizes = pack(streams)
        org = dev(np.asarray(origins, np.int32))
        dims = dev(np.array([[w, h]] * 3, np.int32))
        for flags in (0, 1):
            assert np.array_equal(ctx.decode_region(s, 3, 1, rw - 3, rh - 1, flags),
                                  ctx.decode_region_scaled(s, 1, 3, 1, rw - 3, rh - 1, flags))
            a = torch.full((3, rh, rw, nch), 91, dtype=torch.uint8, device="cuda")
            b = torch.full((3, rh, rw, nch), 91, dtype=torch.uint8, device="cuda")
            ka = kernels_of(ctx, lambda: ctx.decode_batch_region(himg, offs, sizes, w, h, nch, org, rw, rh, flags, out=a))
            kb = kernels_of(ctx, lambda: ctx.decode_batch_region_scaled(himg, offs, sizes, w, h, nch, 1, org, rw, rh, flags, out=b))
            assert ka == kb, (ka, kb)
            _, sa = ctx.decode_batch_region(himg, offs, sizes, w, h, nch, org, rw, rh, flags, out=a)
            _, sb = ctx.decode_batch_region_scaled(himg, offs, sizes, w, h, nch, 1, org, rw, rh, flags, out=b)
            assert torch.equal(sa, sb) and torch.equal(a, b), f"{w}x{h}x{nch} flags {flags}"
            ka = kernels_of(ctx, lambda: ctx.decode_batch_region_mixed(himg, offs, sizes, dims, nch, org, rw, rh, w, h, flags, out=a))
            kb = kernels_of(ctx, lambda: ctx.decode_batch_region_mixed_scaled(himg, offs, sizes, dims, nch, 1, org, rw, rh, w, h,
                                                                              flags, out=b))
            assert ka == kb, (ka, kb)
            _, sa = ctx.decode_batch_region_mixed(himg, offs, sizes, dims, nch, org, rw, rh, w, h, flags, out=a)
            _, sb = ctx.decode_batch_region_mixed_scaled(himg, offs, sizes, dims, nch, 1, org, rw, rh, w, h, flags, out=b)
            assert torch.equal(sa, sb) and torch.equal(a, b), f"mixed {w}x{h}x{nch} flags {flags}"


@gpu
@pytest.mark.parametrize("w, h, nch", [(1920, 1080, 3), (301, 77, 4), (1024, 1024, 1), (37, 21, 6)])
def test_uniform_batch_equals_mixed(ctx, port, w, h, nch):
    streams = [stream(port, w, h, nch, 50, True, k)[0] for k in range(4)] + [b"RIFF" + b"\1" * 40]
    n = len(streams)
    rng = np.random.default_rng(5)
    for f in FACTORS:
        sw, sh = cdiv(w, f), cdiv(h, f)
        rw, rh = max(1, sw // 3), max(1, sh // 2)
        origins = np.stack([rng.integers(0, sw - rw + 1, n), rng.integers(0, sh - rh + 1, n)], 1)
        for flags in (0, 1):
            a, sa, ua = run_batch(ctx, streams, w, h, nch, f, origins, rw, rh, flags)
            b, sb, ub = run_batch(ctx, streams, w, h, nch, f, origins, rw, rh, flags, mixed_dims=[(w, h)] * n, max_wh=(w, h))
            assert ua and ub and list(sa) == list(sb) and sa[4] == REJECT, (f, flags, sa, sb)
            for k in range(4):
                if sa[k] == OK:
                    assert_same(b[k], a[k], f"{w}x{h}x{nch} f {f} flags {flags} image {k}")


def big_image(w, h, nch, seed=5):
    """A smooth seeded [h][w][nch] image with a little noise, made on the device."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.arange(w, dtype=torch.int32, device="cuda").view(1, w, 1)
    y = torch.arange(h, dtype=torch.int32, device="cuda").view(-1, 1, 1)
    k = torch.arange(nch, dtype=torch.int32, device="cuda").view(1, 1, nch)
    v = ((x >> 5) + (y >> 4) * 3 + k * 50 + seed * 17) % 200 + torch.randint(0, 12, (h, w, nch), generator=g, device="cuda",
                                                                             dtype=torch.int32)
    return v.to(torch.uint8)


@gpu
def test_large_batch_equals_scaled_crop(ctx):
    """512 x 1080p: the batch equals decode_batch_scaled cropped on the device."""
    w, h, nch, n = 1920, 1080, 3, 512
    px = torch.stack([big_image(w, h, nch, s) for s in range(8)])
    out, sizes = ctx.encode_batch(px, 50, True)
    ctx.encode_status()
    del px
    idx = torch.arange(n, device="cuda") % 8
    himg = out.reshape(-1)
    offs = idx.to(torch.int64) * out.stride(0)
    sizes = sizes[idx].contiguous()
    rng = np.random.default_rng(1)
    for f, crop in ((2, 224), (4, 224), (8, 112)):
        sw, sh = w // f, h // f
        origins = np.stack([rng.integers(0, sw - crop + 1, n), rng.integers(0, sh - crop + 1, n)], 1).astype(np.int32)
        got, st = ctx.decode_batch_region_scaled(himg, offs, sizes, w, h, nch, f, dev(origins), crop, crop)
        full, fst = ctx.decode_batch_scaled(himg, offs, sizes, w, h, nch, f)
        assert int(st.abs().sum()) == 0 and int(fst.abs().sum()) == 0
        for i in range(n):
            x, y = origins[i]
            assert torch.equal(got[i], full[i, y: y + crop, x: x + crop]), f"f {f} image {i}"
        del full


# ---------------------------------------------------------------------------------------------
# mixed batches
# ---------------------------------------------------------------------------------------------
SIZES = [(64, 48), (40, 24), (37, 21), (96, 64), (500, 300), (512, 300), (8, 8), (1, 1), (1032, 40), (2056, 16),
         (136, 264), (264, 136), (64, 40), (100, 37), (48, 24), (1920, 1080)]


@gpu
@pytest.mark.parametrize("nch", [1, 3, 4])
def test_mixed_matches_oracle(ctx, port, nch):
    streams = [stream(port, w, h, nch)[0] for (w, h) in SIZES]
    wants = [stream(port, w, h, nch)[1] for (w, h) in SIZES]
    rng = np.random.default_rng(3)
    for f in FACTORS:
        for (rw, rh) in ((1, 1), (7, 5), (56, 56)):
            fit = [k for k, (w, h) in enumerate(SIZES) if cdiv(w, f) >= rw and cdiv(h, f) >= rh]
            if not fit:
                continue
            dims = [SIZES[k] for k in fit]
            origins = [(int(rng.integers(0, cdiv(w, f) - rw + 1)), int(rng.integers(0, cdiv(h, f) - rh + 1))) for (w, h) in dims]
            for flags in (0, 1):
                imgs, status, untouched = run_batch(ctx, [streams[k] for k in fit], 0, 0, nch, f, origins, rw, rh, flags,
                                                    mixed_dims=dims, max_wh=(2056, 1080))
                assert untouched
                for j, k in enumerate(fit):
                    want = wants[k][(flags, f)]
                    assert status[j] == (OK if want is not None else REJECT), (f, rw, rh, flags, SIZES[k])
                    if want is not None:
                        x, y = origins[j]
                        assert_same(imgs[j], want[y: y + rh, x: x + rw], f"f {f} {rw}x{rh} flags {flags} image {SIZES[k]}")
                if flags == 1:
                    perm = rng.permutation(len(fit))
                    pimgs, pstatus, _ = run_batch(ctx, [streams[fit[p]] for p in perm], 0, 0, nch, f, [origins[p] for p in perm],
                                                  rw, rh, flags, mixed_dims=[dims[p] for p in perm], max_wh=(2056, 1080))
                    assert list(pstatus) == list(status[perm])
                    assert_same(pimgs, imgs[perm], f"permuted f {f} {rw}x{rh}")
                    for j in range(0, len(fit), 5):  # batches of one
                        one, st, _ = run_batch(ctx, [streams[fit[j]]], 0, 0, nch, f, [origins[j]], rw, rh, flags,
                                               mixed_dims=[dims[j]], max_wh=(2056, 1080))
                        assert st[0] == status[j] and (st[0] != OK or np.array_equal(one[0], imgs[j]))


# ---------------------------------------------------------------------------------------------
# errors
# ---------------------------------------------------------------------------------------------
@gpu
def test_argument_errors(ctx, port):
    import himg_b200

    s, wants = stream(port, 96, 64, 3)
    himg, offs, sizes = pack([s, s])
    org = dev(np.zeros((2, 2), np.int32))
    dims = dev(np.array([[96, 64]] * 2, np.int32))
    out = torch.full((2 * 96 * 64 * 3,), FILL, dtype=torch.uint8, device="cuda")
    status = torch.full((2,), 77, dtype=torch.int32, device="cuda")
    lib, p = ctx.lib, lambda t: C.c_void_p(t.data_ptr())
    buf = np.frombuffer(s, np.uint8)
    host = np.full(96 * 64 * 3, FILL, np.uint8)
    W, H, N = C.c_int(), C.c_int(), C.c_int()

    def single(factor, x, y, rw, rh, cap=host.size):
        return lib.himgcu_decode_region_scaled(ctx.h, buf.ctypes.data, buf.size, 0, factor, x, y, rw, rh, host.ctypes.data, cap,
                                               C.byref(W), C.byref(H), C.byref(N))

    def batch(factor, rw, rh):
        return lib.himgcu_decode_batch_region_scaled(ctx.h, p(himg), p(offs), p(sizes), 2, 96, 64, 3, 0, factor, p(org), rw, rh,
                                                     p(out), p(status))

    def mixed(factor, rw, rh):
        return lib.himgcu_decode_batch_region_mixed_scaled(ctx.h, p(himg), p(offs), p(sizes), 2, p(dims), 96, 64, 3, 0, factor,
                                                           p(org), rw, rh, p(out), p(status))

    for bad in (0, 3, 5, 16, -2):
        assert single(bad, 0, 0, 4, 4) == ERR_ARG and batch(bad, 4, 4) == ERR_ARG and mixed(bad, 4, 4) == ERR_ARG, bad
        with pytest.raises(himg_b200.HimgError) as e:
            ctx.decode_region_scaled(s, bad, 0, 0, 4, 4)
        assert e.value.code == ERR_ARG
    for f in (2, 4, 8):
        sw, sh = 96 // f, 64 // f
        for (x, y, rw, rh) in ((0, 0, sw + 1, 1), (0, 0, 1, sh + 1), (0, 0, 0, 1), (0, 0, 1, 0), (-1, 0, 1, 1), (0, -1, 1, 1),
                               (sw - 3, 0, 4, 1), (0, sh - 1, 1, 2)):
            assert single(f, x, y, rw, rh) == ERR_ARG, (f, x, y, rw, rh)
        for (rw, rh) in ((sw + 1, 1), (1, sh + 1), (0, 1), (1, 0)):
            assert batch(f, rw, rh) == ERR_ARG and mixed(f, rw, rh) == ERR_ARG, (f, rw, rh)
        assert (host == FILL).all()
        # out_cap: the rectangle's size exactly, then one byte less
        need = 5 * 3 * 3
        assert single(f, 1, 2, 5, 3, need - 1) == ERR_CAPACITY
        assert (host == FILL).all()
        assert single(f, 1, 2, 5, 3, need) == OK and (W.value, H.value, N.value) == (96, 64, 3)
        assert_same(host[:need].reshape(3, 5, 3), wants[(0, f)][2:5, 1:6], f"single f {f}")
        assert (host[need:] == FILL).all()
        host[:] = FILL
    ctx.synchronize()
    assert (out.cpu().numpy() == FILL).all() and list(status.cpu().numpy()) == [77, 77], "an argument error wrote something"
    for fn in (lambda n: lib.himgcu_decode_batch_region_scaled(ctx.h, p(himg), p(offs), p(sizes), n, 96, 64, 3, 0, 2, p(org), 4, 4,
                                                               p(out), p(status)),
               lambda n: lib.himgcu_decode_batch_region_mixed_scaled(ctx.h, p(himg), p(offs), p(sizes), n, p(dims), 96, 64, 3, 0, 2,
                                                                     p(org), 4, 4, p(out), p(status))):
        assert fn(-1) == ERR_ARG and fn(0) == OK
    ctx.synchronize()
    assert (out.cpu().numpy() == FILL).all() and list(status.cpu().numpy()) == [77, 77], "n = 0 wrote something"
    with pytest.raises(ValueError):
        ctx.decode_batch_region_scaled(himg, offs, sizes, 96, 64, 3, 2, org.to(torch.int64), 4, 4)
    with pytest.raises(ValueError):
        ctx.decode_batch_region_mixed_scaled(himg, offs, sizes, dims[:1], 3, 2, org, 4, 4, 96, 64)


@gpu
def test_per_image_errors(ctx, port):
    """Origins outside an image's scaled shape and mixed dims out of bounds: ERR_ARG for that image only, its output left
    at the sentinel, its neighbours exact."""
    a, wa = stream(port, 500, 300, 3)
    b, wb = stream(port, 96, 64, 3)
    for f in FACTORS:
        rw, rh = 8 // f + 3, 2
        entries = [  # (stream, want, dims, origin, status)
            (a, wa, (500, 300), (5, 7), OK),
            (a, wa, (500, 300), (cdiv(500, f) - rw + 1, 0), ERR_ARG),  # one column past the scaled width
            (a, wa, (500, 300), (0, cdiv(300, f) - rh + 1), ERR_ARG),  # one row past the scaled height
            (b, wb, (96, 64), (-1, 0), ERR_ARG),
            (b, wb, (96, 64), (cdiv(96, f) - rw, cdiv(64, f) - rh), OK),  # the bottom right corner
            (b, wb, (600, 64), (0, 0), ERR_ARG),  # dims above the bounds
            (b, wb, (0, 64), (0, 0), ERR_ARG),
            (b, wb, (64, 96), (0, 0), REJECT),  # swapped dims: the FRMT shape disagrees
            (a, wa, (500, 300), (cdiv(500, f) - rw, cdiv(300, f) - rh), OK),
        ]
        streams = [e[0] for e in entries]
        origins = [e[3] for e in entries]
        for flags in (0, 1):
            for mixed in (False, True):
                if mixed:
                    ents = entries
                    imgs, status, untouched = run_batch(ctx, streams, 0, 0, 3, f, origins, rw, rh, flags,
                                                        mixed_dims=[e[2] for e in entries], max_wh=(512, 300))
                else:  # the uniform call on the entries of image a
                    ents = [e for e in entries if e[0] is a]
                    imgs, status, untouched = run_batch(ctx, [a] * len(ents), 500, 300, 3, f, [e[3] for e in ents], rw, rh, flags)
                assert list(status) == [e[4] for e in ents], (f, flags, mixed, list(status))
                assert untouched
                for j, e in enumerate(ents):
                    if e[4] == ERR_ARG:
                        assert (imgs[j] == FILL).all(), f"f {f} mixed {mixed}: ERR_ARG image {j} was written"
                    elif e[4] == OK:
                        x, y = e[3]
                        assert_same(imgs[j], e[1][(flags, f)][y: y + rh, x: x + rw], f"neighbour {j} f {f} mixed {mixed}")


@gpu
def test_rejected_streams(ctx, port):
    """Strict-rejected q0 and garbage: the statuses of decode_batch_region on the source rectangles."""
    q0 = port.encode(port.synth(1920, 1080, 3, 1, 6), 0, True)
    good, wants = stream(port, 1920, 1080, 3)
    streams = [q0, good, b"RIFF" + b"\1" * 40, q0, b"\0" * 64, good]
    n = len(streams)
    himg, offs, sizes = pack(streams)
    for f in FACTORS:
        rw, rh = 200 // f, 120 // f
        origins = [(17 * k % (1920 // f - rw), 9 * k % (1080 // f - rh)) for k in range(n)]
        for flags in (0, 1):
            src = dev(np.asarray([(f * x, f * y) for (x, y) in origins], np.int32))
            _, want_st = ctx.decode_batch_region(himg, offs, sizes, 1920, 1080, 3, src, f * rw, f * rh, flags)
            want_st = list(want_st.cpu().numpy())
            assert want_st == ([REJECT, OK, REJECT, REJECT, REJECT, OK] if flags == 0 else [OK, OK, REJECT, OK, REJECT, OK])
            imgs, status, untouched = run_batch(ctx, streams, 1920, 1080, 3, f, origins, rw, rh, flags)
            assert list(status) == want_st and untouched, (f, flags)
            mimgs, mstatus, untouched = run_batch(ctx, streams, 0, 0, 3, f, origins, rw, rh, flags, mixed_dims=[(1920, 1080)] * n,
                                                  max_wh=(1920, 1080))
            assert list(mstatus) == want_st and untouched, (f, flags)
            for k in (1, 5):
                x, y = origins[k]
                assert_same(imgs[k], wants[(flags, f)][y: y + rh, x: x + rw], f"neighbour {k} f {f} flags {flags}")
                assert_same(mimgs[k], imgs[k], f"mixed neighbour {k} f {f} flags {flags}")
            for k in (0, 2):
                got = ctx.decode_region_scaled(streams[k], f, *origins[k], rw, rh, flags)
                assert (got is None) == (want_st[k] == REJECT), (k, f, flags)


# ---------------------------------------------------------------------------------------------
# rows outside the rectangle
# ---------------------------------------------------------------------------------------------
@gpu
def test_rectangle_above_a_broken_chain(ctx, port):
    img = port.synth(256, 400, 3, 3, 6)
    good = port.encode(img, 50, True)
    want = port.decode(good)
    at = good.index(b"FRES") + 8
    mid = at + (len(good) - at) // 2
    bad = bytearray(good)
    bad[mid: mid + 8192] = b"\xff" * min(8192, len(good) - mid)
    bad = bytes(bad)
    for flags in (0, 1):
        assert ctx.decode(bad, flags) is None
        for f in FACTORS:
            sw, sh = 256 // f, 400 // f
            assert_same(ctx.decode_region_scaled(bad, f, 10 // f, 3 // f, 200 // f, 40 // f, flags),
                        box(want, f)[3 // f: 3 // f + 40 // f, 10 // f: 10 // f + 200 // f], f"above the break, f {f} flags {flags}")
            assert ctx.decode_region_scaled(bad, f, 0, sh - 1, sw, 1, flags) is None
            assert ctx.decode_region_scaled(bad, f, 0, 0, sw, sh, flags) is None


@gpu
def test_random_corruption_agrees_with_the_source_region(ctx, port):
    """Status and pixels of himgcu_decode_region on the source rectangle, pooled."""
    img = port.synth(200, 136, 3, 5, 6)
    good = port.encode(img, 60, True)
    rng = np.random.default_rng(3)
    at = good.index(b"FRES") + 8
    for k in range(20):
        bad = bytearray(good)
        lo = 31 if k % 2 else at
        for pos in rng.integers(lo, len(good), 4):
            bad[int(pos)] = int(rng.integers(0, 256))
        bad = bytes(bad)
        for flags in (0, 1):
            for f in FACTORS:
                sw, sh = cdiv(200, f), cdiv(136, f)
                for (x, y, rw, rh) in [(0, 0, sw, sh), (13 // f, 5 // f, 50 // f, 20 // f), (sw - 7, sh - 3, 7, 3)]:
                    sx, sy = f * x, f * y
                    src = ctx.decode_region(bad, sx, sy, min(f * rw, 200 - sx), min(f * rh, 136 - sy), flags)
                    got = ctx.decode_region_scaled(bad, f, x, y, rw, rh, flags)
                    what = f"case {k} flags {flags} f {f} rect {(x, y, rw, rh)}"
                    assert (got is None) == (src is None), what
                    if src is not None:
                        assert_same(got, box(src, f), what)
                    imgs, status, _ = run_batch(ctx, [bad], 200, 136, 3, f, [(x, y)], rw, rh, flags)
                    assert status[0] == (REJECT if src is None else OK), what + " batch"
                    if src is not None:
                        assert_same(imgs[0], box(src, f), what + " batch")


# ---------------------------------------------------------------------------------------------
# calls
# ---------------------------------------------------------------------------------------------
@gpu
def test_sub_batches_and_a_side_stream(port):
    import himg_b200

    sizes_ = [(256, 136), (100, 37), (264, 136), (64, 48), (136, 100), (200, 120), (96, 64), (256, 80), (70, 50)]
    streams = [stream(port, w, h, 3)[0] for (w, h) in sizes_]
    ref = himg_b200.Context(0)
    small = himg_b200.Context(0)
    small.set_option("max_workspace_bytes", 1 << 20)
    rng = np.random.default_rng(2)
    try:
        for f in FACTORS:
            rw, rh = 48 // f, 24 // f
            origins = [(int(rng.integers(0, cdiv(w, f) - rw + 1)), int(rng.integers(0, cdiv(h, f) - rh + 1))) for (w, h) in sizes_]
            want, wst, _ = run_batch(ref, streams, 0, 0, 3, f, origins, rw, rh, 1, mixed_dims=sizes_, max_wh=(264, 136))
            for k, (w, h) in enumerate(sizes_):
                x, y = origins[k]
                assert_same(want[k], stream(port, w, h, 3)[1][(1, f)][y: y + rh, x: x + rw], f"f {f} image {k}")
            got, gst, untouched = run_batch(small, streams, 0, 0, 3, f, origins, rw, rh, 1, mixed_dims=sizes_, max_wh=(264, 136))
            assert untouched and list(gst) == list(wst) and np.array_equal(got, want), f"sub-batches, f {f}"
            same = [stream(port, 264, 136, 3, 50, True, k)[0] for k in range(9)]
            a, sa, _ = run_batch(ref, same, 264, 136, 3, f, origins, rw, rh, 1)
            b, sb, _ = run_batch(small, same, 264, 136, 3, f, origins, rw, rh, 1)
            assert list(sa) == list(sb) == [OK] * 9 and np.array_equal(a, b), f"uniform sub-batches, f {f}"
            side = torch.cuda.Stream()
            with torch.cuda.stream(side):
                c, sc, _ = run_batch(ref, same, 264, 136, 3, f, origins, rw, rh, 1)
            torch.cuda.synchronize()
            assert list(sc) == [OK] * 9 and np.array_equal(c, a), f"side stream, f {f}"
    finally:
        ref.close()
        small.close()


@gpu
def test_viewer_tile_of_a_large_image(ctx):
    """The single-image host call on an 8192^2 gray image: a 1024^2 tile at f = 4, and tiles at the other factors,
    against decode_scaled cropped."""
    w = h = 8192
    out, sizes = ctx.encode_batch(big_image(w, h, 1).unsqueeze(0), 50, True)
    ctx.encode_status()
    data = out[0, : int(sizes[0])].cpu().numpy().tobytes()
    for f, x, y, tw, th in ((4, 512, 768, 1024, 1024), (2, 1000, 3, 1024, 1000), (8, 1, 1, 1023, 1023)):
        full = ctx.decode_scaled(data, f)
        assert_same(ctx.decode_region_scaled(data, f, x, y, tw, th), full[y: y + th, x: x + tw], f"f {f}")
