"""Scaled decode (himgcu_decode_scaled, himgcu_decode_batch_scaled, himgcu_decode_batch_mixed_scaled) against the contract
formula applied to the oracle's decode of each stream.

For a factor f, pixel (y, x, c) of the output is (S + n // 2) // n, where S is the sum of the full decode's channel c over
the f x f window at (f y, f x), clipped to the image, and n the number of its pixels inside the image.  Statuses are
those of the unscaled calls.  Output buffers are filled with a sentinel, so a write outside an image's own output is
seen."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

OK, REJECT, ERR_ARG, ERR_CAPACITY, ERR_UNSUPPORTED = 0, 1, 2, 4, 5
FILL = 0x5A
FACTORS = (1, 2, 4, 8)
# the odd shapes of test_decode_mixed.SIZES, and one shape for every remainder pair of w and h mod 8
ODD = [(1, 1), (17, 3), (37, 21), (300, 5), (2056, 16), (1920, 1080), (3840, 2160)]
REMAINDERS = [(40 + rw, 24 + rh) for rw in range(8) for rh in range(8)]


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
    """A context whose inverse transforms all take the generic (one block per thread) kernels."""
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


def cdiv(a, f):
    return -(-a // f)


_box_memo = {}


def box(d, f):
    """The contract: rounded box averages of d [H][W][C] over f x f windows, clipped at the right and bottom edges."""
    if d is None or f == 1:
        return d
    key = (id(d), f)
    if key not in _box_memo:  # (the memo holds d, so its id is not reused)
        _box_memo[key] = (d, _box(d, f))
    return _box_memo[key][1]


def _box(d, f):
    H, W, nch = d.shape
    oh, ow = cdiv(H, f), cdiv(W, f)
    p = np.zeros((oh * f, ow * f, nch), np.int64)
    p[:H, :W] = d
    s = p.reshape(oh, f, ow, f, nch).sum(axis=(1, 3))
    n = (np.minimum(f, H - f * np.arange(oh))[:, None] * np.minimum(f, W - f * np.arange(ow))[None, :])[..., None]
    return ((s + n // 2) // n).astype(np.uint8)


def box_torch(d, f):
    """box() on the device for [H][W][C] uint8 tensors too large for the host checker, in slabs of block rows."""
    H, W, nch = d.shape
    oh, ow = cdiv(H, f), cdiv(W, f)
    out = torch.empty((oh, ow, nch), dtype=torch.uint8, device=d.device)
    nx = torch.clamp(W - f * torch.arange(ow, device=d.device), max=f).view(1, ow, 1)
    slab = max(1, (1 << 28) // (W * nch * 4 * f))  # output rows per slab
    for y0 in range(0, oh, slab):
        y1 = min(oh, y0 + slab)
        rows = d[f * y0: min(H, f * y1)]
        p = torch.zeros(((y1 - y0) * f, ow * f, nch), dtype=torch.int32, device=d.device)
        p[: rows.shape[0], :W] = rows
        s = p.view(y1 - y0, f, ow, f, nch).sum(dim=(1, 3))
        ny = torch.clamp(H - f * torch.arange(y0, y1, device=d.device), max=f).view(-1, 1, 1)
        n = ny * nx
        out[y0:y1] = torch.div(s + n // 2, n, rounding_mode="floor").to(torch.uint8)
    return out


def pack(streams):
    offs = np.cumsum([0] + [(len(s) + 15) & ~15 for s in streams])
    buf = np.zeros(offs[-1] + 64, np.uint8)
    for o, s in zip(offs, streams):
        buf[o: o + len(s)] = np.frombuffer(s, np.uint8)
    return dev(buf), dev(offs[:-1].astype(np.int64)), dev(np.array([len(s) for s in streams], np.int32))


_streams = {}


def stream(port, w, h, nch, q=50, ycbcr=True, noise=False, seed=None):
    """(stream, strict decode, lenient decode) of the oracle, cached across tests."""
    key = (w, h, nch, q, ycbcr, noise, seed)
    if key not in _streams:
        sd = seed if seed is not None else (w * 7 + h) % 97
        if noise:
            img = np.random.default_rng(sd).integers(0, 256, (h, w, nch), dtype=np.uint8)
        else:
            img = port.synth(w, h, nch, sd, 6)
        s = port.encode(img, q, ycbcr)
        _streams[key] = (s, port.decode(s), port.decode(s, strict=False))
    return _streams[key]


def valid(d, max_w, max_h):
    return 1 <= d[0] <= max_w and 1 <= d[1] <= max_h


def run_batch(c, streams, w, h, nch, f, flags):
    """decode_batch_scaled into a sentinel-filled buffer one image longer than the batch: (images, status, whether the
    spare image kept the sentinel)."""
    n, oh, ow = len(streams), cdiv(h, f), cdiv(w, f)
    out = torch.full((n + 1, oh, ow, nch), FILL, dtype=torch.uint8, device="cuda")
    himg, offs, sizes = pack(streams)
    _, status = c.decode_batch_scaled(himg, offs, sizes, w, h, nch, f, flags, out=out[:n])
    out = out.cpu().numpy()
    return out[:n], status.cpu().numpy(), bool((out[n] == FILL).all())


def run_mixed(c, streams, dims, nch, max_w, max_h, f, flags=0, gap=13, misalign=3):
    """One decode_batch_mixed_scaled call into a sentinel-filled buffer: image i's span starts `gap` bytes after the
    previous one, the first at byte `misalign`; an image with dims out of bounds gets a 64-byte span.  Returns the images
    (None for dims out of bounds), the status and whether every byte outside the spans of images with valid dims kept
    the sentinel."""
    offs, pos, spans = [], misalign, []
    for (w, h) in dims:
        span = cdiv(w, f) * cdiv(h, f) * nch if valid((w, h), max_w, max_h) else 64
        offs.append(pos)
        spans.append(span)
        pos += span + gap
    out = torch.full((pos + 64,), FILL, dtype=torch.uint8, device="cuda")
    himg, o, sizes = pack(streams)
    _, _, status = c.decode_batch_mixed_scaled(himg, o, sizes, dev(np.asarray(dims, np.int32).reshape(-1, 2)), nch, max_w,
                                               max_h, f, flags, out=out, pixel_offsets=dev(np.array(offs, np.int64)))
    buf, status = out.cpu().numpy(), status.cpu().numpy()
    imgs, untouched = [], np.ones(buf.size, bool)
    for (w, h), off, span in zip(dims, offs, spans):
        if valid((w, h), max_w, max_h):
            imgs.append(buf[off: off + span].reshape(cdiv(h, f), cdiv(w, f), nch))
            untouched[off: off + span] = False
        else:
            imgs.append(None)
    return imgs, status, bool((buf[untouched] == FILL).all())


def check(imgs, status, wants, f, flags, what):
    for k, want in enumerate(wants):
        want = want[flags]
        assert status[k] == (OK if want is not None else REJECT), f"{what} image {k}"
        if want is not None:
            assert_same(imgs[k], box(want, f), f"{what} image {k}")


# ---------------------------------------------------------------------------------------------
# every factor on the odd shapes, every channel count, YCbCr on and off, both flag modes
# ---------------------------------------------------------------------------------------------
CHANNELS = [(1, True), (2, True), (3, True), (3, False), (4, True), (4, False), (5, True), (5, False), (6, True), (6, False)]


@pytest.mark.parametrize("nch, ycbcr", CHANNELS)
def test_odd_shapes_match_oracle(ctx, port, nch, ycbcr):
    for (w, h) in ODD:
        s, strict, lenient = stream(port, w, h, nch, 50, ycbcr)
        for f in FACTORS:
            for flags, want in ((0, strict), (1, lenient)):
                what = f"{w}x{h}x{nch} ycbcr {ycbcr} f {f} flags {flags}"
                got = ctx.decode_scaled(s, f, flags)
                assert (got is None) == (want is None), what
                if want is not None:
                    assert_same(got, box(want, f), what + " single")
                imgs, status, untouched = run_batch(ctx, [s, s], w, h, nch, f, flags)
                assert untouched, what + ": written past the batch"
                check(imgs, status, [(strict, lenient)] * 2, f, flags, what + " batch")
        _streams.pop((w, h, nch, 50, ycbcr, False, None))  # (the 4K decodes are large)
        _box_memo.clear()


@pytest.mark.parametrize("nch", [1, 3, 4, 6])
def test_every_remainder_mod_8(ctx, port, nch):
    """All 64 remainder pairs of w and h mod 8 in one mixed batch, and each through decode_batch_scaled."""
    streams = [stream(port, w, h, nch)[0] for (w, h) in REMAINDERS]
    wants = [stream(port, w, h, nch)[1:] for (w, h) in REMAINDERS]
    for f in FACTORS:
        for flags in (0, 1):
            imgs, status, untouched = run_mixed(ctx, streams, REMAINDERS, nch, 47, 31, f, flags)
            assert untouched, f"nch {nch} f {f} flags {flags}: a byte outside the spans was written"
            check(imgs, status, wants, f, flags, f"mixed nch {nch} f {f} flags {flags}")
        for (w, h), s, want in zip(REMAINDERS, streams, wants):
            imgs, status, untouched = run_batch(ctx, [s], w, h, nch, f, 1)
            assert untouched
            check(imgs, status, [want], f, 1, f"batch {w}x{h}x{nch} f {f}")


@pytest.mark.parametrize("q, noise", [(0, False), (50, False), (100, False), (100, True)])
def test_qualities(ctx, generic, port, q, noise):
    """q0 (strict-rejected), q50 and q100 on lane-pair and generic shapes; noise at q100 drives the lane-pair kernel
    into its int32 redo.  The generic kernel gives the same bytes on the lane-pair shapes."""
    for (w, h, nch) in [(1920, 1080, 3), (1024, 64, 1), (256, 136, 3), (300, 77, 3), (37, 21, 1)]:
        s, strict, lenient = stream(port, w, h, nch, q, True, noise)
        for f in FACTORS[1:]:
            for flags, want in ((0, strict), (1, lenient)):
                what = f"{w}x{h}x{nch} q{q} noise {noise} f {f} flags {flags}"
                for c in (ctx, generic):
                    imgs, status, untouched = run_batch(c, [s], w, h, nch, f, flags)
                    assert untouched, what
                    check(imgs, status, [(strict, lenient)], f, flags, what)
                got = ctx.decode_scaled(s, f, flags)
                assert (got is None) == (want is None), what
                if want is not None:
                    assert_same(got, box(want, f), what + " single")


# ---------------------------------------------------------------------------------------------
# the lane-pair kernel against the generic one, and which kernel runs
# ---------------------------------------------------------------------------------------------
def kernels_of(c, fn):
    c.profile(True)
    c.profile_reset()
    try:
        fn()
        c.synchronize()
        return set(c.profile_results())
    finally:
        c.profile(False)


@pytest.mark.parametrize("w, h, nch", [(1920, 1080, 3), (3840, 2160, 3), (1024, 1024, 1), (256, 8, 1), (128, 8, 3)])
def test_lane_pair_equals_generic(ctx, generic, port, w, h, nch):
    s = stream(port, w, h, nch, 70)[0]
    himg, offs, sizes = pack([s] * 3)
    fl = 1  # (lenient: the strict decoder refuses the unframed FRES chunk of an image of one block row)
    for f in FACTORS[1:]:
        k = kernels_of(ctx, lambda: ctx.decode_batch_scaled(himg, offs, sizes, w, h, nch, f, fl))
        assert "k_inverse4_scaled" in k and "k_inverse_scaled" not in k and "k_inverse" not in k, k
        k = kernels_of(generic, lambda: generic.decode_batch_scaled(himg, offs, sizes, w, h, nch, f, fl))
        assert "k_inverse_scaled" in k and "k_inverse4_scaled" not in k, k
        a, sa = ctx.decode_batch_scaled(himg, offs, sizes, w, h, nch, f, fl)
        b, sb = generic.decode_batch_scaled(himg, offs, sizes, w, h, nch, f, fl)
        assert torch.equal(sa, sb) and int(sa.abs().sum()) == 0
        assert torch.equal(a, b), f"{w}x{h}x{nch} f {f}: lane-pair and generic kernels differ"
        # an output offset that is only aligned to the lane-pair kernel's store width of 16 / f bytes
        out = torch.full((3 * (h // f) * (w // f) * nch + 16 // f,), FILL, dtype=torch.uint8, device="cuda")
        view = out[16 // f:].view(3, h // f, w // f, nch)
        k = kernels_of(ctx, lambda: ctx.decode_batch_scaled(himg, offs, sizes, w, h, nch, f, fl, out=view))
        assert "k_inverse4_scaled" in k, k
        assert torch.equal(view, a) and bool((out[: 16 // f] == FILL).all())
    ctx.set_option("xform_variant", 1)
    try:
        k = kernels_of(ctx, lambda: ctx.decode_batch_scaled(himg, offs, sizes, w, h, nch, 2, fl))
        assert "k_inverse_scaled" in k and "k_inverse4_scaled" not in k, k
    finally:
        ctx.set_option("xform_variant", 0)


# ---------------------------------------------------------------------------------------------
# f = 1 is the unscaled call
# ---------------------------------------------------------------------------------------------
def test_factor_one_is_the_unscaled_call(ctx, port):
    garbage = b"RIFF" + b"\1" * 40
    q0 = port.encode(port.synth(264, 136, 3, 1, 6), 0, True)
    for (w, h, nch) in [(1920, 1080, 3), (37, 21, 5), (264, 136, 3)]:
        s = stream(port, w, h, nch)[0]
        for flags in (0, 1):
            a, b = ctx.decode(s, flags), ctx.decode_scaled(s, 1, flags)
            assert (a is None) == (b is None) and (a is None or np.array_equal(a, b)), f"{w}x{h}x{nch} flags {flags}"
            assert flags == 0 or a is not None
            streams = [s, garbage, s] + ([q0] if (w, h, nch) == (264, 136, 3) else [])
            himg, offs, sizes = pack(streams)
            n = len(streams)
            a = torch.full((n, h, w, nch), 91, dtype=torch.uint8, device="cuda")
            b = torch.full((n, h, w, nch), 91, dtype=torch.uint8, device="cuda")
            _, sa = ctx.decode_batch(himg, offs, sizes, w, h, nch, flags, out=a)
            _, sb = ctx.decode_batch_scaled(himg, offs, sizes, w, h, nch, 1, flags, out=b)
            assert torch.equal(sa, sb) and torch.equal(a, b), f"{w}x{h}x{nch} flags {flags}"
            dims = dev(np.array([[w, h]] * n, np.int32))
            a = torch.full((n * w * h * nch + 5,), 91, dtype=torch.uint8, device="cuda")
            b = torch.full((n * w * h * nch + 5,), 91, dtype=torch.uint8, device="cuda")
            po = torch.arange(n, dtype=torch.int64, device="cuda") * (w * h * nch) + 5
            _, _, sa = ctx.decode_batch_mixed(himg, offs, sizes, dims, nch, w, h, flags, out=a, pixel_offsets=po)
            _, _, sb = ctx.decode_batch_mixed_scaled(himg, offs, sizes, dims, nch, w, h, 1, flags, out=b, pixel_offsets=po)
            assert torch.equal(sa, sb) and torch.equal(a, b), f"mixed {w}x{h}x{nch} flags {flags}"
    for data in (garbage, q0):
        for flags in (0, 1):
            a, b = ctx.decode(data, flags), ctx.decode_scaled(data, 1, flags)
            assert (a is None) == (b is None) and (a is None or np.array_equal(a, b))
    assert ctx.decode_scaled(garbage, 2) is None


# ---------------------------------------------------------------------------------------------
# mixed batches
# ---------------------------------------------------------------------------------------------
MIXED_SIZES = [(500, 300), (37, 21), (1920, 1080), (264, 136), (96, 64), (1032, 40), (64, 48), (17, 3), (1, 1), (300, 5)]


def test_mixed_default_offsets_and_allocation(ctx, port):
    streams = [stream(port, w, h, 3)[0] for (w, h) in MIXED_SIZES]
    himg, offs, lens = pack(streams)
    dims = dev(np.array(MIXED_SIZES, np.int32))
    for f in FACTORS[1:]:
        out, px_off, status = ctx.decode_batch_mixed_scaled(himg, offs, lens, dims, 3, 1920, 1080, f, 1)
        spans = [cdiv(w, f) * cdiv(h, f) * 3 for (w, h) in MIXED_SIZES]
        assert out.numel() == sum(spans)
        assert list(px_off.cpu().numpy()) == list(np.cumsum([0] + spans[:-1]))
        assert list(status.cpu().numpy()) == [OK] * len(MIXED_SIZES)
        buf = out.cpu().numpy()
        for k, ((w, h), o) in enumerate(zip(MIXED_SIZES, px_off.cpu().numpy())):
            want = box(stream(port, w, h, 3)[2], f)
            assert_same(buf[o: o + spans[k]].reshape(want.shape), want, f"f {f} image {k}")


def test_mixed_permuted_and_single_images(ctx, port):
    streams = [stream(port, w, h, 3)[0] for (w, h) in MIXED_SIZES]
    wants = [stream(port, w, h, 3)[1:] for (w, h) in MIXED_SIZES]
    rng = np.random.default_rng(11)
    for f in FACTORS[1:]:
        for flags in (0, 1):
            imgs, status, untouched = run_mixed(ctx, streams, MIXED_SIZES, 3, 1920, 1080, f, flags)
            check(imgs, status, wants, f, flags, f"f {f} flags {flags}")
            assert untouched
            perm = rng.permutation(len(MIXED_SIZES))
            pimgs, pstatus, untouched = run_mixed(ctx, [streams[p] for p in perm], [MIXED_SIZES[p] for p in perm], 3, 1920,
                                                  1080, f, flags)
            assert list(pstatus) == list(status[perm]) and untouched
            check(pimgs, pstatus, [wants[p] for p in perm], f, flags, f"permuted, f {f} flags {flags}")
        for k in range(len(MIXED_SIZES)):  # a batch of one
            one, st, untouched = run_mixed(ctx, [streams[k]], [MIXED_SIZES[k]], 3, 1920, 1080, f, 1)
            assert untouched
            check(one, st, [wants[k]], f, 1, f"image {k} alone, f {f}")


@pytest.mark.parametrize("case", [(1920, 1080, 3), (301, 77, 4), (1024, 1024, 1), (37, 21, 6)])
def test_mixed_uniform_batch_equals_batch_scaled(ctx, port, case):
    w, h, nch = case
    streams = [stream(port, w, h, nch, 50, True, False, k)[0] for k in range(4)] + [b"RIFF" + b"\1" * 40]
    himg, offs, sizes = pack(streams)
    n = len(streams)
    for f in FACTORS[1:]:
        img = cdiv(w, f) * cdiv(h, f) * nch
        for flags in (0, 1):
            want_px = torch.full((n, cdiv(h, f), cdiv(w, f), nch), 91, dtype=torch.uint8, device="cuda")
            got_px = torch.full((n * img,), 91, dtype=torch.uint8, device="cuda")
            _, want_st = ctx.decode_batch_scaled(himg, offs, sizes, w, h, nch, f, flags, out=want_px)
            _, _, got_st = ctx.decode_batch_mixed_scaled(
                himg, offs, sizes, dev(np.array([[w, h]] * n, np.int32)), nch, w, h, f, flags, out=got_px,
                pixel_offsets=torch.arange(n, dtype=torch.int64, device="cuda") * img)
            st = list(want_st.cpu().numpy())
            assert list(got_st.cpu().numpy()) == st and st[4] == REJECT and (flags == 0 or st[:4] == [OK] * 4)
            got, want = got_px.cpu().numpy().reshape(n, -1), want_px.cpu().numpy().reshape(n, -1)
            for k in range(4):  # (a rejected image's pixels are unspecified)
                if st[k] == OK:
                    assert_same(got[k], want[k], f"{case} f {f} flags {flags} image {k}")


def test_mixed_per_image_errors(ctx, port):
    nch, max_w, max_h = 3, 512, 300
    a, b = stream(port, 500, 300, nch), stream(port, 96, 64, nch)
    entries = [
        (a, (500, 300), OK),
        (b, (600, 64), ERR_ARG),   # width above the bound
        (b, (96, 301), ERR_ARG),   # height above the bound
        (b, (0, 64), ERR_ARG),     # zero width
        (b, (96, -64), ERR_ARG),   # negative height
        (b, (96, 64), OK),
        (b, (64, 96), REJECT),     # swapped dims: the FRMT shape disagrees
        (a, (96, 64), REJECT),
        (stream(port, 96, 64, 4), (96, 64), REJECT),  # another channel count
        (a, (500, 300), OK),
    ]
    streams = [e[0][0] for e in entries]
    dims = [e[1] for e in entries]
    for f in FACTORS:
        for flags in (0, 1):
            imgs, status, untouched = run_mixed(ctx, streams, dims, nch, max_w, max_h, f, flags)
            assert list(status) == [e[2] for e in entries], f"f {f} flags {flags}"
            assert untouched, f"f {f} flags {flags}: an ERR_ARG span, a gap or a span of no image was written"
            for k, e in enumerate(entries):
                if e[2] == OK:
                    assert_same(imgs[k], box(e[0][1 + flags], f), f"neighbour {k} f {f} flags {flags}")


# ---------------------------------------------------------------------------------------------
# rejected streams: the unscaled call's status, neighbours intact
# ---------------------------------------------------------------------------------------------
def test_rejected_streams(ctx, port):
    q0 = port.encode(port.synth(1920, 1080, 3, 1, 6), 0, True)
    q0_lenient = port.decode(q0, strict=False)
    good, good_strict, good_lenient = stream(port, 1920, 1080, 3)
    streams = [q0, good, b"RIFF" + b"\1" * 40, q0, b"\0" * 64, good]
    himg, offs, sizes = pack(streams)
    n = len(streams)
    for flags in (0, 1):
        _, want_st = ctx.decode_batch(himg, offs, sizes, 1920, 1080, 3, flags)
        want_st = list(want_st.cpu().numpy())
        assert want_st == ([REJECT, OK, REJECT, REJECT, REJECT, OK] if flags == 0 else [OK, OK, REJECT, OK, REJECT, OK])
        for f in FACTORS[1:]:
            imgs, status, untouched = run_batch(ctx, streams, 1920, 1080, 3, f, flags)
            assert list(status) == want_st and untouched, f"f {f} flags {flags}"
            for k in (1, 5):
                assert_same(imgs[k], box(good_lenient if flags else good_strict, f), f"neighbour {k} f {f} flags {flags}")
            if flags:
                assert_same(imgs[0], box(q0_lenient, f), f"lenient q0 f {f}")
            mimgs, mstatus, untouched = run_mixed(ctx, streams, [(1920, 1080)] * n, 3, 1920, 1080, f, flags)
            assert list(mstatus) == want_st and untouched, f"mixed f {f} flags {flags}"
            for k in (1, 5):
                assert_same(mimgs[k], imgs[k], f"mixed neighbour {k} f {f} flags {flags}")
            for k, data in enumerate(streams):
                if k in (1, 2, 3):
                    got = ctx.decode_scaled(data, f, flags)
                    assert (got is None) == (want_st[k] == REJECT), f"single {k} f {f} flags {flags}"


# ---------------------------------------------------------------------------------------------
# host-side argument checks
# ---------------------------------------------------------------------------------------------
def test_argument_errors(ctx, port):
    import himg_b200

    s, strict, _ = stream(port, 96, 64, 3)
    himg, offs, sizes = pack([s, s])
    dims = dev(np.array([[96, 64]] * 2, np.int32))
    px_off = dev(np.array([0, 48 * 32 * 3], np.int64))
    out = torch.full((2 * 96 * 64 * 3,), FILL, dtype=torch.uint8, device="cuda")
    status = torch.full((2,), 77, dtype=torch.int32, device="cuda")
    lib, p = ctx.lib, lambda t: C.c_void_p(t.data_ptr())
    buf = np.frombuffer(s, np.uint8)
    host = np.full(96 * 64 * 3, FILL, np.uint8)
    W, H, N = C.c_int(), C.c_int(), C.c_int()

    def single(factor, cap, data=buf, dst=host):
        return lib.himgcu_decode_scaled(ctx.h, None if data is None else data.ctypes.data, buf.size, 0, factor,
                                        None if dst is None else dst.ctypes.data, cap, C.byref(W), C.byref(H), C.byref(N))

    batch = [C.c_void_p(himg.data_ptr()), p(offs), p(sizes), 2, 96, 64, 3, 0, 2, C.c_void_p(out.data_ptr()), p(status)]
    mixed = [C.c_void_p(himg.data_ptr()), p(offs), p(sizes), 2, p(dims), 96, 64, 3, 0, 2, p(px_off), C.c_void_p(out.data_ptr()),
             p(status)]
    for bad in (0, 3, 5, 16, -2):
        assert single(bad, host.size) == ERR_ARG, bad
        a = list(batch)
        a[8] = bad
        assert lib.himgcu_decode_batch_scaled(ctx.h, *a) == ERR_ARG, bad
        a = list(mixed)
        a[9] = bad
        assert lib.himgcu_decode_batch_mixed_scaled(ctx.h, *a) == ERR_ARG, bad
        with pytest.raises(himg_b200.HimgError) as e:
            ctx.decode_scaled(s, bad)
        assert e.value.code == ERR_ARG
    # out_cap: the scaled size exactly, then one byte less
    for f in FACTORS:
        need = cdiv(96, f) * cdiv(64, f) * 3
        host[:] = FILL
        assert single(f, need - 1) == ERR_CAPACITY, f
        assert (host == FILL).all()
        assert single(f, need) == OK and (W.value, H.value, N.value) == (96, 64, 3)
        assert_same(host[:need].reshape(cdiv(64, f), cdiv(96, f), 3), box(strict, f), f"single f {f}")
        assert (host[need:] == FILL).all()
    assert single(2, host.size, data=None) == ERR_ARG and single(2, host.size, dst=None) == ERR_ARG
    assert lib.himgcu_decode_scaled(None, buf.ctypes.data, buf.size, 0, 2, host.ctypes.data, host.size, None, None, None) == ERR_ARG
    ctx.synchronize()
    out.fill_(FILL)
    for k in (0, 1, 2, 9, 10):  # each pointer of the batch call null in turn
        a = list(batch)
        a[k] = None
        assert lib.himgcu_decode_batch_scaled(ctx.h, *a) == ERR_ARG, k
    for k in (0, 1, 2, 4, 10, 11, 12):
        a = list(mixed)
        a[k] = None
        assert lib.himgcu_decode_batch_mixed_scaled(ctx.h, *a) == ERR_ARG, k
    for call, args, ni in ((lib.himgcu_decode_batch_scaled, batch, 3), (lib.himgcu_decode_batch_mixed_scaled, mixed, 3)):
        a = list(args)
        a[ni] = -1
        assert call(ctx.h, *a) == ERR_ARG
        a[ni] = 0
        assert call(ctx.h, *a) == OK
    ctx.synchronize()
    assert (out.cpu().numpy() == FILL).all() and list(status.cpu().numpy()) == [77, 77], "an error or n = 0 wrote something"
    for (w, h, nch) in [(0, 64, 3), (96, 0, 3), (96, 64, 0), (96, 64, 256), (1 << 16, 1 << 16, 3)]:
        with pytest.raises(himg_b200.HimgError) as e:
            ctx.decode_batch_scaled(himg, offs, sizes, w, h, nch, 2, out=out, status=status)
        assert e.value.code == ERR_UNSUPPORTED, (w, h, nch)
        with pytest.raises(himg_b200.HimgError) as e:
            ctx.decode_batch_mixed_scaled(himg, offs, sizes, dims, nch, w, h, 2, out=out, pixel_offsets=px_off, status=status)
        assert e.value.code == ERR_UNSUPPORTED, (w, h, nch)
    ctx.synchronize()
    assert (out.cpu().numpy() == FILL).all() and list(status.cpu().numpy()) == [77, 77]
    with pytest.raises(ValueError):
        ctx.decode_batch_mixed_scaled(himg, offs, sizes, dims.to(torch.int64), 3, 96, 64, 2)
    with pytest.raises(ValueError):
        ctx.decode_batch_mixed_scaled(himg, offs, sizes, dims, 3, 96, 64, 2, pixel_offsets=px_off[:1])


# ---------------------------------------------------------------------------------------------
# about 2^31 pixel bytes, output offsets past 2^32
# ---------------------------------------------------------------------------------------------
def big_image(w, h, nch):
    """A smooth seeded [h][w][nch] image with a little noise, made on the device in slabs of rows."""
    g = torch.Generator(device="cuda").manual_seed(5)
    img = torch.empty((h, w, nch), dtype=torch.uint8, device="cuda")
    x = torch.arange(w, dtype=torch.int32, device="cuda").view(1, w, 1)
    k = torch.arange(nch, dtype=torch.int32, device="cuda").view(1, 1, nch)
    for y0 in range(0, h, 2048):
        y1 = min(h, y0 + 2048)
        y = torch.arange(y0, y1, dtype=torch.int32, device="cuda").view(-1, 1, 1)
        v = ((x >> 5) + (y >> 4) * 3 + k * 50) % 200 + torch.randint(0, 12, (y1 - y0, w, nch), generator=g, device="cuda",
                                                                     dtype=torch.int32)
        img[y0:y1] = v.to(torch.uint8)
    return img


@pytest.mark.parametrize("w, h, nch, kernel", [
    (46336, 46336, 1, "k_inverse4_scaled"),  # the lane-pair kernel
    (26753, 26753, 3, "k_inverse_scaled"),   # the generic kernel, clipped edge windows
])
def test_near_the_pixel_limit(ctx, w, h, nch, kernel):
    """f = 2 against the pooled decode_batch output.  The lane-pair case decodes ten copies, so that the last image starts
    past 2^32 output bytes; the generic case writes its image at a caller offset past 2^32 (mixed call)."""
    assert w * h * nch < (1 << 31)
    f, oh, ow = 2, cdiv(h, 2), cdiv(w, 2)
    out, sizes = ctx.encode_batch(big_image(w, h, nch).unsqueeze(0), 50, True)
    ctx.encode_status()
    himg = out.reshape(-1)
    full, st = ctx.decode_batch(himg, torch.zeros(1, dtype=torch.int64, device="cuda"), sizes, w, h, nch)
    assert int(st[0]) == OK
    want = box_torch(full[0], f)
    del full
    torch.cuda.empty_cache()
    span = oh * ow * nch
    if nch == 1:
        n = 10
        assert (n - 1) * span > (1 << 32)
        offs = torch.zeros(n, dtype=torch.int64, device="cuda")
        k = kernels_of(ctx, lambda: ctx.decode_batch_scaled(himg, offs[:1], sizes, w, h, nch, f))
        assert kernel in k, k
        got, st = ctx.decode_batch_scaled(himg, offs, sizes.repeat(n), w, h, nch, f)
        assert list(st.cpu().numpy()) == [OK] * n
        for i in (0, n - 1):
            assert torch.equal(got[i], want), f"image {i}"
    else:
        base = (1 << 32) + 3
        buf = torch.full((base + span + 64,), FILL, dtype=torch.uint8, device="cuda")
        dims = torch.tensor([[w, h]], dtype=torch.int32, device="cuda")
        offs = torch.zeros(1, dtype=torch.int64, device="cuda")
        k = kernels_of(ctx, lambda: ctx.decode_batch_mixed_scaled(
            himg, offs, sizes, dims, nch, w, h, f, out=buf, pixel_offsets=torch.tensor([base], device="cuda")))
        assert kernel in k, k
        assert torch.equal(buf[base: base + span].view(oh, ow, nch), want)
        assert bool((buf[base + span:] == FILL).all()) and bool((buf[base - 64: base] == FILL).all())
        got, st = ctx.decode_batch_scaled(himg, offs, sizes, w, h, nch, f)
        assert int(st[0]) == OK and torch.equal(got[0], want)
