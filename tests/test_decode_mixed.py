"""Whole-image decode of mixed-shape batches (himgcu_decode_batch_mixed) against the oracle's decode of each stream,
and against the single-image and same-shape decode calls.

Image i of a mixed batch must give what himgcu_decode gives on its stream alone: the oracle's decode for every stream
it accepts, byte for byte, and the same status otherwise.  The output buffer is filled with a sentinel and the spans
are laid out with gaps, so that a write outside an image's own span is seen."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

# the odd shapes of the region tests, heights of one block row (one unframed FRES segment), and two frame sizes
SIZES = [(64, 48), (40, 24), (37, 21), (96, 64), (500, 300), (512, 300), (8, 8), (1, 1), (1032, 40), (2056, 16),
         (136, 264), (264, 136), (64, 40), (100, 37), (48, 24), (40, 8), (17, 3), (300, 5), (1920, 1080), (3840, 2160)]

OK, REJECT, ERR_ARG, ERR_UNSUPPORTED = 0, 1, 2, 5
FILL = 0x5A


@pytest.fixture(scope="module")
def ctx():
    import himg_b200

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    c = himg_b200.Context(0)
    c.set_stream(torch.cuda.current_stream().cuda_stream)
    yield c
    c.close()


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def assert_same(got, want, what):
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, f"{what}: shape {got.shape} vs {want.shape}"
    idx = np.flatnonzero(got.reshape(-1) != want.reshape(-1))
    assert idx.size == 0, f"{what}: {idx.size} diffs, first at {int(idx[0])}"


def pack(streams):
    offs = np.cumsum([0] + [(len(s) + 15) & ~15 for s in streams])
    buf = np.zeros(offs[-1] + 64, np.uint8)
    for o, s in zip(offs, streams):
        buf[o: o + len(s)] = np.frombuffer(s, np.uint8)
    return dev(buf), dev(offs[:-1].astype(np.int64)), dev(np.array([len(s) for s in streams], np.int32))


_streams = {}


def stream(port, w, h, nch, q=50, seed=None):
    """(stream, strict decode, lenient decode), cached across tests."""
    key = (w, h, nch, q, seed)
    if key not in _streams:
        s = port.encode(port.synth(w, h, nch, seed if seed is not None else (w * 7 + h) % 97, 6), q, True)
        _streams[key] = (s, port.decode(s), port.decode(s, strict=False))
    return _streams[key]


def valid(d, max_w, max_h):
    return 1 <= d[0] <= max_w and 1 <= d[1] <= max_h


def run_mixed(c, streams, dims, nch, max_w, max_h, flags=0, gap=13, misalign=3):
    """One decode_batch_mixed call into a sentinel-filled buffer: image i's span starts `gap` bytes after the previous
    one, the first at byte `misalign`; an image with dims out of bounds gets a 64-byte span.  Returns the images
    ([h][w][nch] arrays, None for dims out of bounds), the status and whether every byte outside the spans of images
    with valid dims kept the sentinel (ERR_ARG spans included)."""
    offs, pos, spans = [], misalign, []
    for (w, h) in dims:
        span = w * h * nch if valid((w, h), max_w, max_h) else 64
        offs.append(pos)
        spans.append(span)
        pos += span + gap
    out = torch.full((pos + 64,), FILL, dtype=torch.uint8, device="cuda")
    himg, o, sizes = pack(streams)
    _, _, status = c.decode_batch_mixed(himg, o, sizes, dev(np.asarray(dims, np.int32).reshape(-1, 2)), nch, max_w, max_h,
                                        flags, out=out, pixel_offsets=dev(np.array(offs, np.int64)))
    buf, status = out.cpu().numpy(), status.cpu().numpy()
    imgs, untouched = [], np.ones(buf.size, bool)
    for (w, h), off, span in zip(dims, offs, spans):
        if valid((w, h), max_w, max_h):
            imgs.append(buf[off: off + span].reshape(h, w, nch))
            untouched[off: off + span] = False
        else:
            imgs.append(None)
    return imgs, status, bool((buf[untouched] == FILL).all())


def check(imgs, status, wants, flags, what):
    for k, want in enumerate(wants):
        want = want[flags]
        assert status[k] == (OK if want is not None else REJECT), f"{what} image {k}"
        if want is not None:
            assert_same(imgs[k], want, f"{what} image {k}")


# ---------------------------------------------------------------------------------------------
# mixed shapes, every channel count, both flag modes
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nch", [1, 2, 3, 4, 5, 6])
def test_mixed_shapes_match_oracle(ctx, port, nch):
    max_w, max_h = max(w for w, _ in SIZES), max(h for _, h in SIZES)
    streams, wants = [], []
    for (w, h) in SIZES:
        s, strict, lenient = stream(port, w, h, nch)
        streams.append(s)
        wants.append((strict, lenient))
    for flags in (0, 1):
        for gap, misalign in ((13, 3), (0, 0)):  # (packed spans from 0 give some images 8-byte aligned rows)
            imgs, status, untouched = run_mixed(ctx, streams, SIZES, nch, max_w, max_h, flags, gap, misalign)
            check(imgs, status, wants, flags, f"nch {nch} flags {flags} gap {gap}")
            assert untouched, f"nch {nch} flags {flags}: a byte outside the spans was written"


def test_default_offsets_and_allocation(ctx, port):
    sizes = [(500, 300), (37, 21), (1920, 1080), (8, 8), (264, 136)]
    streams = [stream(port, w, h, 3)[0] for (w, h) in sizes]
    himg, offs, lens = pack(streams)
    dims = dev(np.array(sizes, np.int32))
    out, px_off, status = ctx.decode_batch_mixed(himg, offs, lens, dims, 3, 1920, 1080, 1)
    spans = [w * h * 3 for (w, h) in sizes]
    assert out.numel() == sum(spans)
    assert list(px_off.cpu().numpy()) == list(np.cumsum([0] + spans[:-1]))
    assert list(status.cpu().numpy()) == [OK] * len(sizes)
    buf = out.cpu().numpy()
    for k, ((w, h), o) in enumerate(zip(sizes, px_off.cpu().numpy())):
        assert_same(buf[o: o + spans[k]].reshape(h, w, 3), stream(port, w, h, 3)[2], f"image {k}")


# ---------------------------------------------------------------------------------------------
# the same-shape call, permutations, single images
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", [(1920, 1080, 3), (301, 77, 4), (1024, 1024, 1)])
def test_uniform_batch_equals_batch(ctx, port, case):
    w, h, nch = case
    streams = [stream(port, w, h, nch, 50, k)[0] for k in range(5)] + [b"RIFF" + b"\1" * 40]
    himg, offs, sizes = pack(streams)
    n, img = len(streams), w * h * nch
    for flags in (0, 1):
        want_px = torch.full((n, h, w, nch), 91, dtype=torch.uint8, device="cuda")
        got_px = torch.full((n * img,), 91, dtype=torch.uint8, device="cuda")
        _, want_st = ctx.decode_batch(himg, offs, sizes, w, h, nch, flags, out=want_px)
        _, _, got_st = ctx.decode_batch_mixed(himg, offs, sizes, dev(np.array([[w, h]] * n, np.int32)), nch, w, h, flags,
                                              out=got_px, pixel_offsets=torch.arange(n, dtype=torch.int64, device="cuda") * img)
        assert list(got_st.cpu().numpy()) == list(want_st.cpu().numpy())
        assert list(got_st.cpu().numpy()) == [OK] * 5 + [REJECT]
        assert_same(got_px.cpu().numpy(), want_px.cpu().numpy().reshape(-1), f"{case} flags {flags}")


def test_permuted_batch_and_single_images(ctx, port):
    sizes = [(500, 300), (37, 21), (1920, 1080), (264, 136), (96, 64), (1032, 40), (64, 48)]
    streams = [stream(port, w, h, 3)[0] for (w, h) in sizes]
    wants = [stream(port, w, h, 3)[1:] for (w, h) in sizes]
    rng = np.random.default_rng(11)
    for flags in (0, 1):
        imgs, status, untouched = run_mixed(ctx, streams, sizes, 3, 1920, 1080, flags)
        check(imgs, status, wants, flags, f"flags {flags}")
        assert untouched
        perm = rng.permutation(len(sizes))
        pimgs, pstatus, untouched = run_mixed(ctx, [streams[p] for p in perm], [sizes[p] for p in perm], 3, 1920, 1080, flags)
        assert list(pstatus) == list(status[perm]) and untouched
        check(pimgs, pstatus, [wants[p] for p in perm], flags, f"permuted, flags {flags}")
        for k in range(len(sizes)):  # a batch of one (its low-res branch runs beside the segment table)
            one, st, untouched = run_mixed(ctx, [streams[k]], [sizes[k]], 3, 1920, 1080, flags)
            assert list(st) == [status[k]] and untouched
            check(one, st, [wants[k]], flags, f"image {k} alone, flags {flags}")


# ---------------------------------------------------------------------------------------------
# both variants of the FRES stream decoder
# ---------------------------------------------------------------------------------------------
def decode_team(streams, out_bytes, base=32):
    """Threads per stream that the library's decode_team gives (api.cu)."""
    team = base
    while team < 1024 and streams * team < 131072 and out_bytes // (team * 2) >= 256:
        team *= 2
    return team


@pytest.mark.parametrize("case", ["warp_teams", "wide_teams", "wide_teams_single"])
def test_both_stream_decoders(ctx, port, case):
    if case == "warp_teams":  # 32 images of 1080p bounds: 32 * 135 block rows fill the GPU with one warp per row
        sizes = [(1920, 1080), (1000, 700), (37, 21), (1032, 40)] * 8
        max_w, max_h = 1920, 1080
    elif case == "wide_teams":  # three images of 4K bounds: few block rows, wide teams
        sizes = [(3840, 2160), (2000, 1500), (500, 300)]
        max_w, max_h = 3840, 2160
    else:  # one image: also the forked low-res branch
        sizes = [(3840, 2160)]
        max_w, max_h = 3840, 2160
    rows, seg = (max_h + 7) // 8, (max_w + 7) // 8 * 64 * 3
    team = decode_team(len(sizes) * rows, seg)
    assert (team == 32) == (case == "warp_teams"), team
    streams = [stream(port, w, h, 3)[0] for (w, h) in sizes]
    wants = [stream(port, w, h, 3)[1:] for (w, h) in sizes]
    for flags in (0, 1):
        imgs, status, untouched = run_mixed(ctx, streams, sizes, 3, max_w, max_h, flags)
        check(imgs, status, wants, flags, f"{case} flags {flags}")
        assert untouched
    if len(sizes) > 1:  # (a profiled single image does not fork, so the batch of one runs unprofiled above)
        ctx.profile(True)
        ctx.profile_reset()
        try:
            run_mixed(ctx, streams, sizes, 3, max_w, max_h, 1)
            ctx.synchronize()
            assert ctx.profile_results()["k_dec_stream_fres"][1] == 1
        finally:
            ctx.profile(False)


# ---------------------------------------------------------------------------------------------
# per-image errors and rejections
# ---------------------------------------------------------------------------------------------
def test_per_image_errors(ctx, port):
    nch, max_w, max_h = 3, 512, 300
    a, b = stream(port, 500, 300, nch), stream(port, 96, 64, nch)
    entries = [
        (a, (500, 300), OK),
        (b, (600, 64), ERR_ARG),   # width above the bound
        (b, (96, 301), ERR_ARG),   # height above the bound
        (b, (0, 64), ERR_ARG),     # zero width
        (b, (96, 0), ERR_ARG),     # zero height
        (b, (-5, 64), ERR_ARG),    # negative width
        (b, (96, -64), ERR_ARG),   # negative height
        (b, (96, 64), OK),
        (b, (64, 96), REJECT),     # swapped dims: the FRMT shape disagrees
        (b, (88, 64), REJECT),
        (a, (96, 64), REJECT),
        (stream(port, 96, 64, 4), (96, 64), REJECT),  # another channel count
        (a, (500, 300), OK),
    ]
    streams = [e[0][0] for e in entries]
    dims = [e[1] for e in entries]
    for flags in (0, 1):
        imgs, status, untouched = run_mixed(ctx, streams, dims, nch, max_w, max_h, flags)
        assert list(status) == [e[2] for e in entries], f"flags {flags}"
        assert untouched, f"flags {flags}: an ERR_ARG span, a gap or a span of no image was written"
        for k, e in enumerate(entries):
            if e[2] == OK:
                assert_same(imgs[k], e[0][1 + flags], f"neighbour {k} flags {flags}")


def test_strict_rejects_q0_and_garbage(ctx, port):
    q0 = port.encode(port.synth(1920, 1080, 3, 1, 6), 0, True)
    assert port.decode(q0) is None
    want = port.decode(q0, strict=False)
    good, good_want, _ = stream(port, 264, 136, 3)
    streams = [q0, good, b"RIFF" + b"\1" * 40, q0, b"\0" * 64]
    dims = [(1920, 1080), (264, 136), (300, 64), (1920, 1080), (256, 64)]
    for flags in (0, 1):
        imgs, status, untouched = run_mixed(ctx, streams, dims, 3, 1920, 1080, flags)
        assert untouched
        if flags == 0:
            assert list(status) == [REJECT, OK, REJECT, REJECT, REJECT]
        else:
            assert list(status) == [OK, OK, REJECT, OK, REJECT]
            assert_same(imgs[0], want, "lenient q0 image 0")
            assert_same(imgs[3], want, "lenient q0 image 3")
        assert_same(imgs[1], good_want, f"neighbour flags {flags}")


def test_random_corruption_agrees_with_single_image(ctx, port):
    rng = np.random.default_rng(7)
    sizes = [(200, 136), (37, 21), (512, 300), (64, 48)]
    streams, dims = [], []
    for k in range(20):
        w, h = sizes[k % len(sizes)]
        good = stream(port, w, h, 3, 60)[0]
        bad = bytearray(good)
        lo = 31 if k % 2 else good.index(b"FRES") + 8
        for pos in rng.integers(lo, len(good), 4):
            bad[int(pos)] = int(rng.integers(0, 256))
        streams.append(bytes(bad))
        dims.append((w, h))
    for flags in (0, 1):
        imgs, status, untouched = run_mixed(ctx, streams, dims, 3, 512, 300, flags)
        assert untouched, f"flags {flags}"
        for k in range(20):
            single = ctx.decode(streams[k], flags)
            assert status[k] == (OK if single is not None else REJECT), f"case {k} flags {flags}"
            if single is not None:
                assert_same(imgs[k], single, f"case {k} flags {flags}")


# ---------------------------------------------------------------------------------------------
# round trip with the mixed encoder
# ---------------------------------------------------------------------------------------------
def test_round_trip_with_encode_batch_mixed(ctx, port):
    sizes = [(500, 300), (37, 21), (1920, 1080), (8, 8), (264, 136), (1032, 40), (17, 3)]
    imgs = [port.synth(w, h, 3, 40 + k, 6) for k, (w, h) in enumerate(sizes)]
    offs, pos = [], 5
    for im in imgs:
        offs.append(pos)
        pos += im.size + 7
    buf = np.zeros(pos, np.uint8)
    for o, im in zip(offs, imgs):
        buf[o: o + im.size] = im.reshape(-1)
    pixels, px_off, dims = dev(buf), dev(np.array(offs, np.int64)), dev(np.array(sizes, np.int32))
    out, lens = ctx.encode_batch_mixed(pixels, px_off, dims, 3, 1920, 1080, 50, True)
    n = len(sizes)
    offsets = torch.arange(n, dtype=torch.int64, device="cuda") * out.stride(0)
    rows = out.cpu().numpy()
    for flags in (0, 1):
        dec = torch.full((pos,), FILL, dtype=torch.uint8, device="cuda")
        _, _, status = ctx.decode_batch_mixed(out.reshape(-1), offsets, lens, dims, 3, 1920, 1080, flags, out=dec,
                                              pixel_offsets=px_off)
        status, got = status.cpu().numpy(), dec.cpu().numpy()
        for k, ((w, h), o) in enumerate(zip(sizes, offs)):
            want = port.decode(rows[k, : int(lens[k])].tobytes(), strict=not flags)
            assert status[k] == (OK if want is not None else REJECT), f"image {k} flags {flags}"
            if want is not None:
                assert_same(got[o: o + w * h * 3].reshape(h, w, 3), want, f"image {k} flags {flags}")


# ---------------------------------------------------------------------------------------------
# sub-batches, streams, host-side argument checks
# ---------------------------------------------------------------------------------------------
def test_sub_batches(port):
    import himg_b200

    sizes = [(256, 136), (100, 37), (264, 136), (64, 48), (136, 100), (200, 120), (96, 64), (256, 80), (70, 50)]
    streams = [stream(port, w, h, 3)[0] for (w, h) in sizes]
    wants = [stream(port, w, h, 3)[1:] for (w, h) in sizes]
    c = himg_b200.Context(0)
    try:
        n0 = c.launch_count()
        run_mixed(c, streams, sizes, 3, 264, 136, 1)
        one = c.launch_count() - n0
        c.set_option("max_workspace_bytes", 1 << 20)
        n0 = c.launch_count()
        imgs, status, untouched = run_mixed(c, streams, sizes, 3, 264, 136, 1)
        assert c.launch_count() - n0 >= 3 * one, "the batch was not split"
        assert untouched
        check(imgs, status, wants, 1, "sub-batched")
    finally:
        c.close()


def test_on_a_side_stream(port):
    import himg_b200

    sizes = [(512, 304), (300, 200), (640, 480), (256, 256), (1032, 40), (200, 500)]
    streams = [stream(port, w, h, 3)[0] for (w, h) in sizes]
    offs = np.cumsum([0] + [(len(s) + 15) & ~15 for s in streams])
    buf = np.zeros(offs[-1] + 64, np.uint8)
    for o, s in zip(offs, streams):
        buf[o: o + len(s)] = np.frombuffer(s, np.uint8)
    c = himg_b200.Context(0)
    try:
        s = torch.cuda.Stream()
        with torch.cuda.stream(s):
            torch.cuda._sleep(20_000_000)  # the inputs arrive late on s
            himg = torch.from_numpy(buf).pin_memory().cuda(non_blocking=True)
            o = torch.from_numpy(offs[:-1].astype(np.int64)).pin_memory().cuda(non_blocking=True)
            sz = torch.from_numpy(np.array([len(x) for x in streams], np.int32)).pin_memory().cuda(non_blocking=True)
            dims = torch.from_numpy(np.array(sizes, np.int32)).pin_memory().cuda(non_blocking=True)
            px, px_off, status = c.decode_batch_mixed(himg, o, sz, dims, 3, 1032, 500, 1)
            total = px.to(torch.int64).sum()
            px_h, off_h = px.cpu(), px_off.cpu()
        s.synchronize()
        assert list(status.cpu().numpy()) == [OK] * len(sizes)
        px_h, off_h = px_h.numpy(), off_h.numpy()
        ref = 0
        for k, (w, h) in enumerate(sizes):
            want = stream(port, w, h, 3)[2]
            assert_same(px_h[off_h[k]: off_h[k] + w * h * 3].reshape(h, w, 3), want, f"side stream image {k}")
            ref += int(want.astype(np.int64).sum())
        assert int(total.cpu()) == ref
    finally:
        c.close()


def test_host_argument_errors(ctx, port):
    import ctypes as C

    import himg_b200

    s = stream(port, 96, 64, 3)[0]
    himg, offs, sizes = pack([s, s])
    dims = dev(np.array([[96, 64]] * 2, np.int32))
    px_off = dev(np.array([0, 96 * 64 * 3], np.int64))
    out = torch.full((2 * 96 * 64 * 3,), FILL, dtype=torch.uint8, device="cuda")
    status = torch.full((2,), 77, dtype=torch.int32, device="cuda")
    for (mw, mh, nch) in [(0, 64, 3), (96, 0, 3), (96, 64, 0), (96, 64, 256), (1 << 16, 1 << 16, 3)]:
        with pytest.raises(himg_b200.HimgError) as e:
            ctx.decode_batch_mixed(himg, offs, sizes, dims, nch, mw, mh, out=out, pixel_offsets=px_off, status=status)
        assert e.value.code == ERR_UNSUPPORTED, (mw, mh, nch)
    lib, p = ctx.lib, lambda t: C.c_void_p(t.data_ptr())
    args = [C.c_void_p(himg.data_ptr()), p(offs), p(sizes), 2, p(dims), 96, 64, 3, 0, p(px_off), C.c_void_p(out.data_ptr()),
            p(status)]
    for k in (0, 1, 2, 4, 9, 10, 11):  # each pointer null in turn
        a = list(args)
        a[k] = None
        assert lib.himgcu_decode_batch_mixed(ctx.h, *a) == ERR_ARG, k
    a = list(args)
    a[3] = -1
    assert lib.himgcu_decode_batch_mixed(ctx.h, *a) == ERR_ARG
    a[3] = 0
    assert lib.himgcu_decode_batch_mixed(ctx.h, *a) == OK
    ctx.synchronize()
    assert (out.cpu().numpy() == FILL).all() and list(status.cpu().numpy()) == [77, 77], "n = 0 wrote something"
    with pytest.raises(ValueError):
        ctx.decode_batch_mixed(himg, offs, sizes, dims.to(torch.int64), 3, 96, 64)
    with pytest.raises(ValueError):
        ctx.decode_batch_mixed(himg, offs, sizes, dims[:1], 3, 96, 64)
    with pytest.raises(ValueError):
        ctx.decode_batch_mixed(himg, offs, sizes, dims, 3, 96, 64, pixel_offsets=px_off.to(torch.int32))
    with pytest.raises(ValueError):
        ctx.decode_batch_mixed(himg, offs, sizes, dims, 3, 96, 64, pixel_offsets=px_off[:1])
