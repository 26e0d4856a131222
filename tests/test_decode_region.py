"""Region decode (himgcu_decode_region / himgcu_decode_batch_region) against the oracle's whole-image decode, cropped.

A region must equal the crop of the whole decode byte for byte, accept every stream the whole decode accepts and
reject only streams the whole decode rejects too."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

SHAPES = [(64, 48, 3), (40, 24, 1), (37, 21, 1), (96, 64, 4), (500, 300, 3), (512, 300, 3), (8, 8, 1), (1, 1, 3),
          (1032, 40, 3), (2056, 16, 1), (136, 264, 2), (264, 136, 4), (64, 40, 5), (100, 37, 6), (48, 24, 8)]

OK, REJECT, ERR_ARG = 0, 1, 2


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


def rects(w, h):
    """Whole image, 1x1 corners, every y % 8 and x % 8 phase, rectangles ending in the partial last block
    row / column, a rectangle inside one block row."""
    out = [(0, 0, w, h), (0, 0, 1, 1), (w - 1, 0, 1, 1), (0, h - 1, 1, 1), (w - 1, h - 1, 1, 1)]
    for p in range(8):
        if p < h:
            out.append((0, p, w, min(h - p, 11)))
        if p < w:
            out.append((p, 0, min(w - p, 13), h))
    out.append((max(0, w - 11), max(0, h - 5), min(w, 11), min(h, 5)))
    out.append((w // 3, h - 1, w - w // 3, 1))
    r = (h // 8) // 2 * 8
    out.append((w // 4, r + 2, max(1, w // 2), min(5, h - r - 2) if h - r - 2 > 0 else 1))
    return [(x, y, rw, rh) for (x, y, rw, rh) in out if rw >= 1 and rh >= 1 and x + rw <= w and y + rh <= h]


def pack(streams):
    offs = np.cumsum([0] + [(len(s) + 15) & ~15 for s in streams])
    buf = np.zeros(offs[-1] + 64, np.uint8)
    for o, s in zip(offs, streams):
        buf[o: o + len(s)] = np.frombuffer(s, np.uint8)
    return dev(buf), dev(offs[:-1].astype(np.int64)), dev(np.array([len(s) for s in streams], np.int32))


# ---------------------------------------------------------------------------------------------
# single image, host call
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("quality", [50, 5])
def test_region_matches_crop(ctx, port, shape, quality):
    w, h, n = shape
    packed = port.encode(port.synth(w, h, n, 4, 6), quality, True)
    for flags in (0, 1):
        want = port.decode(packed, strict=(flags == 0))
        whole = ctx.decode_region(packed, 0, 0, w, h, flags)
        assert (whole is None) == (want is None), f"{shape} q{quality} flags {flags}: reject mismatch"
        if want is None:
            continue
        for (x, y, rw, rh) in rects(w, h):
            got = ctx.decode_region(packed, x, y, rw, rh, flags)
            assert got is not None, f"{shape} region {(x, y, rw, rh)} rejected"
            assert_same(got, want[y: y + rh, x: x + rw], f"{shape} q{quality} flags {flags} region {(x, y, rw, rh)}")


def test_region_bad_rectangles_raise(ctx, port):
    import himg_b200

    packed = port.encode(port.synth(64, 48, 3, 1, 6), 50, True)
    for (x, y, rw, rh) in [(0, 0, 0, 5), (0, 0, 5, 0), (-1, 0, 4, 4), (0, -1, 4, 4), (61, 0, 4, 4), (0, 45, 4, 4),
                           (0, 0, 65, 48), (0, 0, 64, 49)]:
        with pytest.raises(himg_b200.HimgError) as e:
            ctx.decode_region(packed, x, y, rw, rh)
        assert e.value.code == ERR_ARG
    assert ctx.decode_region(b"RIFF" + b"\0" * 20, 0, 0, 1, 1) is None
    assert ctx.decode_region(packed[:-1], 0, 0, 1, 1) is None


def test_region_strict_reject_q0(ctx, port):
    img = port.synth(1920, 1080, 3, 1, 6)
    packed = port.encode(img, 0, True)
    assert port.decode(packed) is None
    want = port.decode(packed, strict=False)
    assert ctx.decode_region(packed, 100, 200, 224, 224) is None
    assert_same(ctx.decode_region(packed, 100, 200, 224, 224, 1), want[200:424, 100:324], "lenient q0 region")
    himg, offs, sizes = pack([packed, packed])
    origins = dev(np.array([[0, 0], [1696, 856]], np.int32))
    for flags in (0, 1):
        px, status = ctx.decode_batch_region(himg, offs, sizes, 1920, 1080, 3, origins, 224, 224, flags)
        status = status.cpu().numpy()
        if flags == 0:
            assert list(status) == [REJECT, REJECT]
        else:
            assert list(status) == [OK, OK]
            px = px.cpu().numpy()
            assert_same(px[0], want[:224, :224], "lenient batch region 0")
            assert_same(px[1], want[856:, 1696:], "lenient batch region 1")


def test_region_above_a_broken_chain(ctx, port):
    # a segment header broken half way down: the whole decode rejects, a region above the break does not read it
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
        assert_same(ctx.decode_region(bad, 10, 3, 200, 40, flags), want[3:43, 10:210], f"region above the break, flags {flags}")
        assert ctx.decode_region(bad, 0, 392, 256, 8, flags) is None
        assert ctx.decode_region(bad, 0, 0, 256, 400, flags) is None


def test_region_random_corruption(ctx, port):
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
            full = ctx.decode(bad, flags)
            for (x, y, rw, rh) in [(0, 0, 200, 136), (13, 5, 50, 20), (150, 100, 50, 36)]:
                got = ctx.decode_region(bad, x, y, rw, rh, flags)
                if full is not None:
                    assert got is not None, f"case {k} flags {flags}: the whole decode accepts, the region rejects"
                    assert_same(got, full[y: y + rh, x: x + rw], f"case {k} flags {flags} region {(x, y, rw, rh)}")


# ---------------------------------------------------------------------------------------------
# batch, device call
# ---------------------------------------------------------------------------------------------
def _batch_case(ctx, port, w, h, n, B, rw, rh, q, seed):
    imgs = [port.synth(w, h, n, seed + k, 6) for k in range(B)]
    streams = [port.encode(im, q, True) for im in imgs]
    wants = [port.decode(s) for s in streams]
    rng = np.random.default_rng(seed)
    origins = np.stack([rng.integers(0, w - rw + 1, B), rng.integers(0, h - rh + 1, B)], 1).astype(np.int32)
    return streams, wants, origins


def _run_batch(ctx, streams, w, h, n, origins, rw, rh, flags=0):
    himg, offs, sizes = pack(streams)
    px, status = ctx.decode_batch_region(himg, offs, sizes, w, h, n, dev(origins), rw, rh, flags)
    return px.cpu().numpy(), status.cpu().numpy()


@pytest.mark.parametrize("case", [(1920, 1080, 3, 8, 224, 224, 50), (301, 77, 4, 5, 40, 30, 60), (1024, 1024, 1, 3, 200, 150, 50)])
@pytest.mark.parametrize("generic", [0, 1])
def test_batch_region(port, case, generic):
    import himg_b200

    w, h, n, B, rw, rh, q = case
    c = himg_b200.Context(0)
    try:
        c.set_option("force_generic", generic)
        streams, wants, origins = _batch_case(c, port, w, h, n, B, rw, rh, q, 17)
        c.profile(True)
        px, status = _run_batch(c, streams, w, h, n, origins, rw, rh)
        c.synchronize()
        names = c.profile_results()
        assert list(status) == [OK] * B
        for k in range(B):
            x, y = origins[k]
            assert_same(px[k], wants[k][y: y + rh, x: x + rw], f"{case} generic={generic} image {k} at {(x, y)}")
        fast = not generic and n in (1, 3) and ((w + 7) // 8) % 16 == 0
        assert ("k_inverse_region4" in names) == fast, names
        assert ("k_inverse_region" in names) == (not fast), names
        assert "k_inverse" not in names
    finally:
        c.close()


def test_batch_region_whole_frame_and_positions(ctx, port):
    # the whole frame as a region, and one stream at several batch positions with the same origin
    w, h, n = 1920, 1080, 3
    a, b = port.encode(port.synth(w, h, n, 1, 6), 50, True), port.encode(port.synth(w, h, n, 2, 6), 50, True)
    want_a = port.decode(a)
    px, status = _run_batch(ctx, [a, b, a, a], w, h, n, np.zeros((4, 2), np.int32), w, h)
    assert list(status) == [OK] * 4
    assert_same(px[0], want_a, "whole frame")
    assert_same(px[1], port.decode(b), "whole frame, image 1")
    origins = np.array([[777, 333]] * 4, np.int32)
    px, status = _run_batch(ctx, [a, b, a, a], w, h, n, origins, 333, 251)
    assert list(status) == [OK] * 4
    for k in (0, 2, 3):
        assert_same(px[k], want_a[333:584, 777:1110], f"position {k}")


def test_batch_region_sub_batches(port):
    import himg_b200

    w, h, n, B, rw, rh = 256, 136, 3, 9, 70, 50
    streams, wants, origins = _batch_case(None, port, w, h, n, B, rw, rh, 50, 40)
    c = himg_b200.Context(0)
    try:
        n0 = c.launch_count()
        _run_batch(c, streams, w, h, n, origins, rw, rh)
        one = c.launch_count() - n0  # launches of an unsplit batch
        c.set_option("max_workspace_bytes", 1 << 20)  # a few images per sub-batch
        n0 = c.launch_count()
        px, status = _run_batch(c, streams, w, h, n, origins, rw, rh)
        assert c.launch_count() - n0 >= 3 * one, "the batch was not split"
        assert list(status) == [OK] * B
        for k in range(B):
            x, y = origins[k]
            assert_same(px[k], wants[k][y: y + rh, x: x + rw], f"sub-batched image {k}")
    finally:
        c.close()


def test_batch_region_rejects_and_bad_origins(ctx, port):
    import himg_b200

    w, h, n, rw, rh = 128, 64, 3, 32, 24
    good = [port.encode(port.synth(w, h, n, k, 6), 50, True) for k in range(3)]
    streams = good + [b"RIFF" + b"\1" * 40, port.encode(port.synth(64, 64, n, 9, 6), 50, True), good[0], good[1], good[2]]
    origins = np.array([[0, 0], [96, 40], [5, 7], [0, 0], [0, 0], [-1, 0], [97, 0], [0, 41]], np.int32)
    himg, offs, sizes = pack(streams)
    out = torch.full((len(streams), rh, rw, n), 77, dtype=torch.uint8, device="cuda")
    px, status = ctx.decode_batch_region(himg, offs, sizes, w, h, n, dev(origins), rw, rh, out=out)
    px, status = px.cpu().numpy(), status.cpu().numpy()
    assert list(status) == [OK, OK, OK, REJECT, REJECT, ERR_ARG, ERR_ARG, ERR_ARG]
    for k in range(3):
        x, y = origins[k]
        assert_same(px[k], port.decode(good[k])[y: y + rh, x: x + rw], f"neighbour {k}")
    assert (px[5:] == 77).all(), "an image with a bad origin was written"
    for (cw, chh) in [(0, 5), (5, 0), (w + 1, 5), (5, h + 1)]:
        with pytest.raises(himg_b200.HimgError):
            ctx.decode_batch_region(himg, offs, sizes, w, h, n, dev(origins), cw, chh)


def test_batch_region_on_a_side_stream(port):
    # the call runs on torch's current stream: ordered after the copies that made its inputs and before the
    # work that reads its output, on a non-default stream
    import himg_b200

    w, h, n, B, rw, rh = 512, 304, 3, 6, 100, 90
    streams, wants, origins = _batch_case(None, port, w, h, n, B, rw, rh, 50, 60)
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
            org = torch.from_numpy(origins).pin_memory().cuda(non_blocking=True)
            px, status = c.decode_batch_region(himg, o, sz, w, h, n, org, rw, rh)
            total = px.to(torch.int64).sum()
            px_h = px.cpu()
        s.synchronize()
        assert list(status.cpu().numpy()) == [OK] * B
        px_h = px_h.numpy()
        ref = 0
        for k in range(B):
            x, y = origins[k]
            crop = wants[k][y: y + rh, x: x + rw]
            assert_same(px_h[k], crop, f"side stream image {k}")
            ref += int(crop.astype(np.int64).sum())
        assert int(total.cpu()) == ref
    finally:
        c.close()
