"""Region decode of mixed-shape batches (himgcu_decode_batch_region_mixed) against the oracle's whole-image decode,
cropped, and against the single-image and same-shape region calls.

Image i of a mixed batch must give what himgcu_decode_region gives on its stream alone: the crop of the whole decode
for every stream the whole decode accepts, byte for byte, and the same status otherwise."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

# the odd shapes of the region tests, and two frame sizes
SIZES = [(64, 48), (40, 24), (37, 21), (96, 64), (500, 300), (512, 300), (8, 8), (1, 1), (1032, 40), (2056, 16),
         (136, 264), (264, 136), (64, 40), (100, 37), (48, 24), (1920, 1080), (3840, 2160)]
CROPS = [(1, 1), (7, 5), (16, 16), (224, 224)]

OK, REJECT, ERR_ARG, ERR_UNSUPPORTED = 0, 1, 2, 5


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


def run_mixed(c, streams, dims, nch, origins, rw, rh, max_w, max_h, flags=0, fill=None):
    himg, offs, sizes = pack(streams)
    out = None
    if fill is not None:
        out = torch.full((len(streams), rh, rw, nch), fill, dtype=torch.uint8, device="cuda")
    px, status = c.decode_batch_region_mixed(himg, offs, sizes, dev(np.asarray(dims, np.int32).reshape(-1, 2)), nch,
                                             dev(np.asarray(origins, np.int32).reshape(-1, 2)), rw, rh, max_w, max_h, flags,
                                             out=out)
    return px.cpu().numpy(), status.cpu().numpy()


def origins_for(w, h, rw, rh):
    """Corners (the last one ends in the partial last block row and column), every x % 8 and y % 8 phase, and the
    rectangle ending in the last block row / column at a phase."""
    xs, ys = w - rw, h - rh
    out = [(0, 0), (xs, 0), (0, ys), (xs, ys)]
    for p in range(8):
        out.append((min(p, xs), min((3 * p + 1) % 8, ys)))
    out.append((max(0, xs - 3), max(0, ys - 5)))
    return list(dict.fromkeys(out))


_streams = {}


def stream(port, w, h, nch, q=50, seed=None):
    """(stream, strict whole decode, lenient whole decode), cached across tests."""
    key = (w, h, nch, q, seed)
    if key not in _streams:
        s = port.encode(port.synth(w, h, nch, seed if seed is not None else (w * 7 + h) % 97, 6), q, True)
        _streams[key] = (s, port.decode(s), port.decode(s, strict=False))
    return _streams[key]


# ---------------------------------------------------------------------------------------------
# mixed shapes, every crop size and origin phase, both flag modes
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nch", [1, 3, 4, 5])
def test_mixed_matches_crops(ctx, port, nch):
    sizes = SIZES
    max_w, max_h = max(w for w, _ in sizes), max(h for _, h in sizes)
    for rw, rh in CROPS:
        streams, dims, origins, wants = [], [], [], []
        for (w, h) in sizes:
            if rw > w or rh > h:
                continue
            s, strict, lenient = stream(port, w, h, nch)
            for (x, y) in origins_for(w, h, rw, rh):
                streams.append(s)
                dims.append((w, h))
                origins.append((x, y))
                wants.append((strict, lenient))
        for flags in (0, 1):
            px, status = run_mixed(ctx, streams, dims, nch, origins, rw, rh, max_w, max_h, flags)
            for k, ((x, y), (w, h), want) in enumerate(zip(origins, dims, wants)):
                want = want[flags]
                what = f"nch {nch} crop {rw}x{rh} flags {flags} image {k} ({w}x{h}) at {(x, y)}"
                assert status[k] == (OK if want is not None else REJECT), what
                if want is not None:
                    assert_same(px[k], want[y: y + rh, x: x + rw], what)


# ---------------------------------------------------------------------------------------------
# the same-shape call, permutations, single images
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", [(1920, 1080, 3, 224, 224), (301, 77, 4, 40, 30), (1024, 1024, 1, 200, 150)])
def test_uniform_batch_equals_batch_region(ctx, port, case):
    w, h, nch, rw, rh = case
    streams = [stream(port, w, h, nch, 50, k)[0] for k in range(5)] + [b"RIFF" + b"\1" * 40]
    rng = np.random.default_rng(5)
    origins = np.stack([rng.integers(0, w - rw + 1, 6), rng.integers(0, h - rh + 1, 6)], 1).astype(np.int32)
    origins[4] = (w - rw + 1, 0)  # outside the image: ERR_ARG
    himg, offs, sizes = pack(streams)
    for flags in (0, 1):
        want_px = torch.full((6, rh, rw, nch), 91, dtype=torch.uint8, device="cuda")
        got_px = torch.full((6, rh, rw, nch), 91, dtype=torch.uint8, device="cuda")
        _, want_st = ctx.decode_batch_region(himg, offs, sizes, w, h, nch, dev(origins), rw, rh, flags, out=want_px)
        _, got_st = ctx.decode_batch_region_mixed(himg, offs, sizes, dev(np.array([[w, h]] * 6, np.int32)), nch, dev(origins),
                                                  rw, rh, w, h, flags, out=got_px)
        assert list(got_st.cpu().numpy()) == list(want_st.cpu().numpy())
        assert list(got_st.cpu().numpy()) == [OK] * 4 + [ERR_ARG, REJECT]
        assert_same(got_px.cpu().numpy(), want_px.cpu().numpy(), f"{case} flags {flags}")


def test_permuted_batch_and_single_images(ctx, port):
    sizes = [(500, 300), (37, 21), (1920, 1080), (264, 136), (96, 64), (1032, 40), (64, 48)]
    rw, rh = 33, 17
    streams = [stream(port, w, h, 3)[0] for (w, h) in sizes]
    rng = np.random.default_rng(11)
    origins = [(int(rng.integers(0, w - rw + 1)), int(rng.integers(0, h - rh + 1))) for (w, h) in sizes]
    # lenient: the strict mode rejects the small images whose FRES chunk is shorter than one block row
    px, status = run_mixed(ctx, streams, sizes, 3, origins, rw, rh, 1920, 1080, 1)
    assert list(status) == [OK] * len(sizes)
    for k, (w, h) in enumerate(sizes):
        x, y = origins[k]
        assert_same(px[k], stream(port, w, h, 3)[2][y: y + rh, x: x + rw], f"image {k}")
    perm = rng.permutation(len(sizes))
    ppx, pstatus = run_mixed(ctx, [streams[p] for p in perm], [sizes[p] for p in perm], 3, [origins[p] for p in perm], rw, rh,
                             1920, 1080, 1)
    assert list(pstatus) == list(status[perm])
    assert_same(ppx, px[perm], "permuted batch")
    for k in range(len(sizes)):  # a batch of one (its low-res branch runs beside the segment table)
        one, st = run_mixed(ctx, [streams[k]], [sizes[k]], 3, [origins[k]], rw, rh, 1920, 1080, 1)
        assert list(st) == [OK]
        assert_same(one[0], px[k], f"image {k} alone")


# ---------------------------------------------------------------------------------------------
# per-image errors and rejections
# ---------------------------------------------------------------------------------------------
def test_per_image_errors(ctx, port):
    rw, rh, nch, max_w, max_h = 24, 16, 3, 512, 300
    a, b, small = stream(port, 500, 300, nch)[0], stream(port, 96, 64, nch)[0], stream(port, 20, 12, nch)[0]
    entries = [
        (a, (500, 300), (3, 5), OK),
        (b, (600, 64), (0, 0), ERR_ARG),   # width above the bound
        (b, (96, 301), (0, 0), ERR_ARG),   # height above the bound
        (b, (0, 64), (0, 0), ERR_ARG),     # zero width
        (b, (96, 0), (0, 0), ERR_ARG),     # zero height
        (b, (-5, 64), (0, 0), ERR_ARG),    # negative width
        (b, (96, 64), (70, 40), OK),
        (b, (88, 64), (0, 0), REJECT),     # dims that disagree with the stream
        (b, (96, 56), (0, 0), REJECT),
        (a, (96, 64), (0, 0), REJECT),
        (small, (20, 12), (0, 0), ERR_ARG),  # the crop is larger than the image
        (b, (96, 64), (73, 0), ERR_ARG),    # origin outside the image
        (b, (96, 64), (0, -1), ERR_ARG),
        (stream(port, 96, 64, 4)[0], (96, 64), (0, 0), REJECT),  # another channel count
        (a, (500, 300), (476, 284), OK),
    ]
    streams = [e[0] for e in entries]
    dims = [e[1] for e in entries]
    origins = [e[2] for e in entries]
    for flags in (0, 1):
        px, status = run_mixed(ctx, streams, dims, nch, origins, rw, rh, max_w, max_h, flags, fill=77)
        assert list(status) == [e[3] for e in entries], f"flags {flags}"
        for k, e in enumerate(entries):
            if e[3] == OK:
                (w, h), (x, y) = e[1], e[2]
                assert_same(px[k], stream(port, w, h, nch)[1 + flags][y: y + rh, x: x + rw], f"neighbour {k} flags {flags}")
            elif e[3] == ERR_ARG:
                assert (px[k] == 77).all(), f"image {k} with status ERR_ARG was written"


def test_strict_rejects_q0_and_garbage(ctx, port):
    q0 = port.encode(port.synth(1920, 1080, 3, 1, 6), 0, True)
    assert port.decode(q0) is None
    want = port.decode(q0, strict=False)
    good, good_want, _ = stream(port, 264, 136, 3)
    streams = [q0, good, b"RIFF" + b"\1" * 40, q0, b"\0" * 64]
    dims = [(1920, 1080), (264, 136), (300, 64), (1920, 1080), (256, 64)]
    origins = [(0, 0), (40, 100), (0, 0), (1696, 856), (0, 0)]
    for flags in (0, 1):
        px, status = run_mixed(ctx, streams, dims, 3, origins, 224, 36, 1920, 1080, flags)
        if flags == 0:
            assert list(status) == [REJECT, OK, REJECT, REJECT, REJECT]
        else:
            assert list(status) == [OK, OK, REJECT, OK, REJECT]
            assert_same(px[0], want[:36, :224], "lenient q0 image 0")
            assert_same(px[3], want[856:892, 1696:], "lenient q0 image 3")
        assert_same(px[1], good_want[100:136, 40:264], f"neighbour flags {flags}")


def test_region_above_a_broken_chain(ctx, port):
    good, want, _ = stream(port, 256, 400, 3, 50, 3)
    at = good.index(b"FRES") + 8
    mid = at + (len(good) - at) // 2
    bad = bytearray(good)
    bad[mid: mid + 8192] = b"\xff" * min(8192, len(good) - mid)
    bad = bytes(bad)
    other, other_want, _ = stream(port, 96, 64, 3)
    streams = [bad, other, bad, bad]
    dims = [(256, 400), (96, 64), (256, 400), (256, 400)]
    origins = [(10, 3), (5, 2), (0, 392), (200, 0)]
    for flags in (0, 1):
        px, status = run_mixed(ctx, streams, dims, 3, origins, 32, 8, 256, 400, flags)
        assert list(status) == [OK, OK, REJECT, OK], f"flags {flags}"
        assert_same(px[0], want[3:11, 10:42], f"region above the break, flags {flags}")
        assert_same(px[1], other_want[2:10, 5:37], f"neighbour, flags {flags}")
        assert_same(px[3], want[0:8, 200:232], f"region above the break, flags {flags}")
        assert ctx.decode_region(bad, 0, 392, 32, 8, flags) is None


def test_random_corruption_agrees_with_single_image_region(ctx, port):
    rng = np.random.default_rng(7)
    sizes = [(200, 136), (37, 21), (512, 300), (64, 48)]
    rw, rh = 30, 20
    streams, dims, origins = [], [], []
    for k in range(20):
        w, h = sizes[k % len(sizes)]
        good = stream(port, w, h, 3, 60)[0]
        bad = bytearray(good)
        lo = 31 if k % 2 else good.index(b"FRES") + 8
        for pos in rng.integers(lo, len(good), 4):
            bad[int(pos)] = int(rng.integers(0, 256))
        streams.append(bytes(bad))
        dims.append((w, h))
        origins.append((int(rng.integers(0, w - rw + 1)), int(rng.integers(0, h - rh + 1))))
    for flags in (0, 1):
        px, status = run_mixed(ctx, streams, dims, 3, origins, rw, rh, 512, 300, flags)
        for k in range(20):
            x, y = origins[k]
            single = ctx.decode_region(streams[k], x, y, rw, rh, flags)
            assert status[k] == (OK if single is not None else REJECT), f"case {k} flags {flags}"
            if single is not None:
                assert_same(px[k], single, f"case {k} flags {flags}")


# ---------------------------------------------------------------------------------------------
# sub-batches, streams, host-side argument checks
# ---------------------------------------------------------------------------------------------
def test_sub_batches(port):
    import himg_b200

    sizes = [(256, 136), (100, 37), (264, 136), (64, 48), (136, 100), (200, 120), (96, 64), (256, 80), (70, 50)]
    rw, rh = 60, 30
    streams = [stream(port, w, h, 3)[0] for (w, h) in sizes]
    rng = np.random.default_rng(2)
    origins = [(int(rng.integers(0, w - rw + 1)), int(rng.integers(0, h - rh + 1))) for (w, h) in sizes]
    c = himg_b200.Context(0)
    try:
        n0 = c.launch_count()
        run_mixed(c, streams, sizes, 3, origins, rw, rh, 264, 136, 1)
        one = c.launch_count() - n0
        c.set_option("max_workspace_bytes", 1 << 20)
        n0 = c.launch_count()
        px, status = run_mixed(c, streams, sizes, 3, origins, rw, rh, 264, 136, 1)
        assert c.launch_count() - n0 >= 3 * one, "the batch was not split"
        assert list(status) == [OK] * len(sizes)
        for k, (w, h) in enumerate(sizes):
            x, y = origins[k]
            assert_same(px[k], stream(port, w, h, 3)[2][y: y + rh, x: x + rw], f"sub-batched image {k}")
    finally:
        c.close()


def test_on_a_side_stream(port):
    import himg_b200

    sizes = [(512, 304), (300, 200), (640, 480), (256, 256), (1032, 40), (200, 500)]
    rw, rh = 100, 40
    streams = [stream(port, w, h, 3)[0] for (w, h) in sizes]
    rng = np.random.default_rng(9)
    origins = np.array([(rng.integers(0, w - rw + 1), rng.integers(0, h - rh + 1)) for (w, h) in sizes], np.int32)
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
            org = torch.from_numpy(origins).pin_memory().cuda(non_blocking=True)
            px, status = c.decode_batch_region_mixed(himg, o, sz, dims, 3, org, rw, rh, 1032, 500, 1)
            total = px.to(torch.int64).sum()
            px_h = px.cpu()
        s.synchronize()
        assert list(status.cpu().numpy()) == [OK] * len(sizes)
        px_h = px_h.numpy()
        ref = 0
        for k, (w, h) in enumerate(sizes):
            x, y = origins[k]
            crop = stream(port, w, h, 3)[2][y: y + rh, x: x + rw]
            assert_same(px_h[k], crop, f"side stream image {k}")
            ref += int(crop.astype(np.int64).sum())
        assert int(total.cpu()) == ref
    finally:
        c.close()


def test_host_argument_errors(ctx, port):
    import himg_b200

    s = stream(port, 96, 64, 3)[0]
    himg, offs, sizes = pack([s, s])
    dims = dev(np.array([[96, 64]] * 2, np.int32))
    origins = dev(np.zeros((2, 2), np.int32))
    for (rw, rh, mw, mh, nch, code) in [(0, 5, 96, 64, 3, ERR_ARG), (5, 0, 96, 64, 3, ERR_ARG), (97, 5, 96, 64, 3, ERR_ARG),
                                        (5, 65, 96, 64, 3, ERR_ARG), (5, 5, 0, 64, 3, ERR_UNSUPPORTED),
                                        (5, 5, 96, 0, 3, ERR_UNSUPPORTED), (5, 5, 96, 64, 256, ERR_UNSUPPORTED),
(5, 5, 1 << 16, 1 << 16, 3, ERR_UNSUPPORTED)]:
        with pytest.raises(himg_b200.HimgError) as e:
            ctx.decode_batch_region_mixed(himg, offs, sizes, dims, nch, origins, rw, rh, mw, mh)
        assert e.value.code == code, (rw, rh, mw, mh, nch)
    with pytest.raises(ValueError):
        ctx.decode_batch_region_mixed(himg, offs, sizes, dims.to(torch.int64), 3, origins, 5, 5, 96, 64)
    with pytest.raises(ValueError):
        ctx.decode_batch_region_mixed(himg, offs, sizes, dims[:1], 3, origins, 5, 5, 96, 64)
    with pytest.raises(ValueError):
        ctx.decode_batch_region_mixed(himg, offs, sizes, dims, 3, origins[:1], 5, 5, 96, 64)
