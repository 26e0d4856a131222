"""Encode of mixed-shape batches (himgcu_encode_batch_mixed) against the oracle's encode of each image alone, and
against the same-shape batch call.

Image i of a mixed batch must give exactly the stream (bytes and size) that himgcu_encode gives for it alone, whatever
the other images of the batch, its position in the batch and where its pixels lie in the input buffer."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

# the odd shapes of the region tests, heights of one block row (one unframed FRES segment), and two frame sizes
SIZES = [(64, 48), (40, 24), (37, 21), (96, 64), (500, 300), (512, 300), (8, 8), (1, 1), (1032, 40), (2056, 16),
         (136, 264), (264, 136), (64, 40), (100, 37), (48, 24), (40, 8), (17, 3), (300, 5), (1920, 1080), (3840, 2160)]
SMALL = [s for s in SIZES if s[0] * s[1] <= 600 * 300]

OK, ERR_ARG, ERR_CAPACITY, ERR_UNSUPPORTED = 0, 2, 4, 5


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


_imgs, _want = {}, {}


def image(port, w, h, nch, seed=None, flat=False):
    key = (w, h, nch, seed, flat)
    if key not in _imgs:
        if flat:  # constant colour: all-zero coefficient planes (zero runs over whole segments)
            _imgs[key] = np.full((h, w, nch), (seed or 0) * 37 % 256, np.uint8)
        else:
            _imgs[key] = port.synth(w, h, nch, seed if seed is not None else (w * 7 + h) % 97, 6)
    return _imgs[key]


def want(port, img, q=50, ycbcr=True):
    key = (img.shape, q, ycbcr, hash(img.tobytes()))
    if key not in _want:
        _want[key] = port.encode(img, q, ycbcr)
    return _want[key]


def pack(imgs, gap=0, misalign=0):
    """One flat device buffer with image i at offsets[i]: `gap` bytes between images, the first at byte `misalign`."""
    offs, pos = [], misalign
    for im in imgs:
        offs.append(pos)
        pos += im.size + gap
    buf = np.full(pos + 64, 0xA5, np.uint8)
    for o, im in zip(offs, imgs):
        buf[o: o + im.size] = im.reshape(-1)
    return dev(buf), dev(np.array(offs, np.int64))


def run_mixed(c, imgs, nch, q=50, ycbcr=True, dims=None, bounds=None, gap=0, misalign=0, out=None):
    """Streams (None where the size is 0), sizes and the output rows of one encode_batch_mixed call."""
    pixels, offs = pack(imgs, gap, misalign)
    if dims is None:
        dims = [(im.shape[1], im.shape[0]) for im in imgs]
    if bounds is None:
        bounds = (max(d[0] for d in dims), max(d[1] for d in dims))
    out, sizes = c.encode_batch_mixed(pixels, offs, dev(np.asarray(dims, np.int32).reshape(-1, 2)), nch, bounds[0], bounds[1],
                                      q, ycbcr, out=out)
    rows, sizes = out.cpu().numpy(), sizes.cpu().numpy()
    return [rows[k, : sizes[k]].tobytes() if sizes[k] else None for k in range(len(imgs))], sizes, rows


def check(streams, imgs, port, q=50, ycbcr=True, what=""):
    for k, (s, im) in enumerate(zip(streams, imgs)):
        w = want(port, im, q, ycbcr)
        assert s is not None, f"{what} image {k} {im.shape}: size 0"
        assert len(s) == len(w), f"{what} image {k} {im.shape}: size {len(s)} vs {len(w)}"
        assert s == w, f"{what} image {k} {im.shape}: first diff at {next(i for i in range(len(w)) if s[i] != w[i])}"


def check_ref(streams, imgs, q=50, ycbcr=True, limit=300 * 300):
    import oracle

    if not oracle.ref_available():
        return
    ref = oracle.ref()
    for k, (s, im) in enumerate(zip(streams, imgs)):
        if im.shape[0] * im.shape[1] <= limit:
            assert s == ref.encode(im, q, ycbcr), f"image {k} {im.shape} differs from the reference"


# ---------------------------------------------------------------------------------------------
# mixed shapes, channel counts, qualities, colour spaces
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nch", [1, 2, 3, 4, 5])
def test_mixed_matches_single_image_encode(ctx, port, nch):
    imgs = [image(port, w, h, nch) for (w, h) in SIZES]
    streams, _, _ = run_mixed(ctx, imgs, nch)
    check(streams, imgs, port, what=f"nch {nch}")
    check_ref(streams, imgs)


@pytest.mark.parametrize("q", [0, 50, 100])
@pytest.mark.parametrize("ycbcr", [True, False])
@pytest.mark.parametrize("nch", [1, 3, 4, 5])
def test_quality_and_colour_space(ctx, port, q, ycbcr, nch):
    imgs = [image(port, w, h, nch, 3) for (w, h) in SMALL]
    streams, _, _ = run_mixed(ctx, imgs, nch, q, ycbcr)
    check(streams, imgs, port, q, ycbcr, f"nch {nch} q {q} ycbcr {ycbcr}")
    check_ref(streams, imgs, q, ycbcr, 200 * 200)


# ---------------------------------------------------------------------------------------------
# both entropy coders of the FRES chunk, with and without item lists
# ---------------------------------------------------------------------------------------------
def coder_variants(port, imgs, nch):
    import himg_b200

    out = {}
    for name, opts in [("default", {}), ("teams", {"huff_warp_teams": 2}), ("ctas", {"huff_warp_teams": 0}),
                       ("no lists", {"item_lists": 0}), ("teams, no lists", {"huff_warp_teams": 2, "item_lists": 0})]:
        c = himg_b200.Context(0)
        try:
            for k, v in opts.items():
                c.set_option(k, v)
            out[name] = run_mixed(c, imgs, nch)[0]
            c.encode_status()
        finally:
            c.close()
    return out


def test_entropy_coders_large_batch(port):
    # 40 images bounded by 1080p: n x 135 block rows >= 148 SMs x 32 warps, so the default codes FRES with warp teams
    rng = np.random.default_rng(3)
    dims = [(1920, 1080)] + [(int(rng.integers(200, 1921)), int(rng.integers(100, 1081))) for _ in range(39)]
    imgs = [image(port, w, h, 3, k) for k, (w, h) in enumerate(dims)]
    res = coder_variants(port, imgs, 3)
    check(res["default"], imgs, port, what="default coder")
    for name, streams in res.items():
        assert streams == res["default"], name


def test_entropy_coders_small_batch(port):
    # six images: the default codes FRES with a CTA per segment
    imgs = [image(port, w, h, 4, 5) for (w, h) in [(500, 300), (37, 21), (264, 136), (1, 1), (40, 8), (1032, 40)]]
    res = coder_variants(port, imgs, 4)
    check(res["default"], imgs, port, what="default coder")
    for name, streams in res.items():
        assert streams == res["default"], name


def test_flat_images(port):
    # constant images: runs of 16 662 zeros and more, and runs of 65 536 and more inside the 4K segments (no item list)
    imgs = [image(port, 3840, 2160, 3, 1, flat=True), image(port, 500, 300, 3), image(port, 1920, 1080, 3, 2, flat=True),
            image(port, 2056, 16, 3, 3, flat=True), image(port, 64, 48, 3, 4, flat=True)]
    half = image(port, 3840, 2160, 3, 9).copy()
    half[:, 1920:] = 200
    imgs.append(half)
    res = coder_variants(port, imgs, 3)
    check(res["default"], imgs, port, what="flat")
    for name, streams in res.items():
        assert streams == res["default"], name


# ---------------------------------------------------------------------------------------------
# the same-shape call, batch layout, sub-batches
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", [(1920, 1080, 3), (301, 77, 4), (1024, 1024, 1), (640, 480, 5)])
def test_uniform_batch_equals_encode_batch(ctx, port, case):
    # encode_batch takes the lane-pair transforms (k_lowres_avg2 / k_forward3) where the shape allows them, the mixed
    # call the generic ones: two independent implementations
    w, h, nch = case
    imgs = [image(port, w, h, nch, k) for k in range(4)]
    px = dev(np.stack(imgs))
    want_out, want_sizes = ctx.encode_batch(px, 50, True)
    streams, sizes, _ = run_mixed(ctx, imgs, nch)
    assert list(sizes) == list(want_sizes.cpu().numpy())
    wo = want_out.cpu().numpy()
    for k in range(4):
        assert streams[k] == wo[k, : sizes[k]].tobytes(), f"image {k}"
    check(streams[:1], imgs[:1], port)


def test_batch_layout(ctx, port):
    sizes = [(500, 300), (37, 21), (1920, 1080), (264, 136), (1, 1), (96, 64), (1032, 40), (17, 3)]
    imgs = [image(port, w, h, 3) for (w, h) in sizes]
    streams, _, _ = run_mixed(ctx, imgs, 3)
    check(streams, imgs, port)
    perm = np.random.default_rng(11).permutation(len(imgs))
    pstreams, _, _ = run_mixed(ctx, [imgs[p] for p in perm], 3)
    assert pstreams == [streams[p] for p in perm], "permuted batch"
    gapped, _, _ = run_mixed(ctx, imgs, 3, gap=5, misalign=3)  # odd offsets, bytes between the images
    assert gapped == streams, "offsets with gaps and odd alignment"
    for k in range(len(imgs)):  # a batch of one, under the bounds of the whole batch
        one, _, _ = run_mixed(ctx, [imgs[k]], 3, bounds=(1920, 1080), misalign=k)
        assert one[0] == streams[k], f"image {k} alone"


def test_sub_batches(port):
    import himg_b200

    sizes = [(256, 136), (100, 37), (264, 136), (64, 48), (136, 100), (200, 120), (96, 64), (256, 80), (70, 50)]
    imgs = [image(port, w, h, 3) for (w, h) in sizes]
    c = himg_b200.Context(0)
    try:
        n0 = c.launch_count()
        whole, _, _ = run_mixed(c, imgs, 3)
        one = c.launch_count() - n0
        c.set_option("max_workspace_bytes", 1 << 20)
        n0 = c.launch_count()
        split, _, _ = run_mixed(c, imgs, 3)
        assert c.launch_count() - n0 >= 3 * one, "the batch was not split"
        assert split == whole
        check(split, imgs, port)
        c.encode_status()
    finally:
        c.close()


# ---------------------------------------------------------------------------------------------
# per-image errors
# ---------------------------------------------------------------------------------------------
def test_per_image_dims_errors(port):
    import himg_b200

    a, b = image(port, 500, 300, 3), image(port, 96, 64, 3)
    entries = [(a, (500, 300), True), (b, (600, 64), False), (b, (96, 301), False), (b, (0, 64), False), (b, (96, 0), False),
               (b, (-5, 64), False), (b, (96, -1), False), (b, (96, 64), True), (a, (500, 300), True)]
    imgs = [e[0] for e in entries]
    c = himg_b200.Context(0)
    try:
        out = torch.full((len(entries), 1 << 20), 77, dtype=torch.uint8, device="cuda")
        streams, sizes, rows = run_mixed(c, imgs, 3, dims=[e[1] for e in entries], bounds=(512, 300), out=out)
        for k, (im, _, good) in enumerate(entries):
            if good:
                check([streams[k]], [im], port, what=f"neighbour {k}")
            else:
                assert sizes[k] == 0 and (rows[k] == 77).all(), f"image {k} with bad dims was written"
        with pytest.raises(himg_b200.HimgError) as e:
            c.encode_status()
        assert e.value.code == ERR_ARG
        c.encode_status()  # (read = clear)
    finally:
        c.close()


def test_per_image_capacity(port):
    import himg_b200

    small, large = [image(port, 64, 48, 3), image(port, 37, 21, 3)], [image(port, 1920, 1080, 3), image(port, 500, 300, 3)]
    imgs = [small[0], large[0], small[1], large[1]]
    stride = 8192  # fits the small streams only
    assert all(len(want(port, im)) <= stride for im in small) and all(len(want(port, im)) > stride for im in large)
    c = himg_b200.Context(0)
    try:
        for bad_dims in (False, True):
            out = torch.full((len(imgs) + 1, stride), 77, dtype=torch.uint8, device="cuda")
            batch = imgs + [small[0]]
            dims = [(im.shape[1], im.shape[0]) for im in imgs] + [(0, 48) if bad_dims else (64, 48)]
            streams, sizes, rows = run_mixed(c, batch, 3, dims=dims, bounds=(1920, 1080), out=out)
            check([streams[0], streams[2]], small, port, what="fits")
            for k in (1, 3):
                assert sizes[k] == 0 and (rows[k] == 77).all(), f"image {k} did not fit but was written"
            with pytest.raises(himg_b200.HimgError) as e:
                c.encode_status()
            assert e.value.code == ERR_CAPACITY, "the capacity error outranks the dims error" if bad_dims else ""
    finally:
        c.close()


# ---------------------------------------------------------------------------------------------
# host-side argument errors, streams, end to end
# ---------------------------------------------------------------------------------------------
def test_host_argument_errors(ctx, port):
    import himg_b200

    im = image(port, 96, 64, 3)
    pixels, offs = pack([im, im])
    dims = dev(np.array([[96, 64]] * 2, np.int32))
    for (mw, mh, nch, code) in [(0, 64, 3, ERR_UNSUPPORTED), (96, 0, 3, ERR_UNSUPPORTED), (96, 64, 0, ERR_UNSUPPORTED),
                                (96, 64, 256, ERR_UNSUPPORTED), (1 << 16, 1 << 16, 3, ERR_UNSUPPORTED)]:
        with pytest.raises(himg_b200.HimgError) as e:
            ctx.encode_batch_mixed(pixels, offs, dims, nch, mw, mh, out=torch.empty((2, 256), dtype=torch.uint8, device="cuda"))
        assert e.value.code == code, (mw, mh, nch)
    out = torch.empty((2, 1 << 16), dtype=torch.uint8, device="cuda")
    sizes = torch.empty((2,), dtype=torch.int32, device="cuda")
    lib, P = ctx.lib, lambda t: t.data_ptr()
    args = [P(pixels), P(offs), P(dims), 2, 96, 64, 3, 50, 1, P(out), out.stride(0), P(sizes)]
    for k in (0, 1, 2, 9, 11):  # null pointers
        a = list(args)
        a[k] = None
        assert lib.himgcu_encode_batch_mixed(ctx.h, *a) == ERR_ARG, k
    a = list(args)
    a[3] = -1
    assert lib.himgcu_encode_batch_mixed(ctx.h, *a) == ERR_ARG
    assert lib.himgcu_encode_batch_mixed(None, *args) == ERR_ARG
    a = list(args)
    a[3] = 0
    assert lib.himgcu_encode_batch_mixed(ctx.h, *a) == OK
    with pytest.raises(ValueError):
        ctx.encode_batch_mixed(pixels, offs, dims.to(torch.int64), 3, 96, 64)
    with pytest.raises(ValueError):
        ctx.encode_batch_mixed(pixels, offs.to(torch.int32), dims, 3, 96, 64)
    with pytest.raises(ValueError):
        ctx.encode_batch_mixed(pixels, offs, dims[:1], 3, 96, 64)
    ctx.encode_status()


def test_on_a_side_stream(port):
    import himg_b200

    sizes = [(512, 304), (300, 200), (640, 480), (256, 256), (1032, 40), (200, 500)]
    imgs = [image(port, w, h, 3) for (w, h) in sizes]
    offs = np.cumsum([0] + [im.size for im in imgs])
    buf = np.concatenate([im.reshape(-1) for im in imgs])
    c = himg_b200.Context(0)
    try:
        s = torch.cuda.Stream()
        with torch.cuda.stream(s):
            torch.cuda._sleep(20_000_000)  # the inputs arrive late on s
            px = torch.from_numpy(buf).pin_memory().cuda(non_blocking=True)
            o = torch.from_numpy(offs[:-1].astype(np.int64)).pin_memory().cuda(non_blocking=True)
            dims = torch.from_numpy(np.array(sizes, np.int32)).pin_memory().cuda(non_blocking=True)
            out, sz = c.encode_batch_mixed(px, o, dims, 3, 1032, 500)
            total = sz.to(torch.int64).sum()
            out_h, sz_h = out.cpu(), sz.cpu()
        s.synchronize()
        out_h, sz_h = out_h.numpy(), sz_h.numpy()
        check([out_h[k, : sz_h[k]].tobytes() for k in range(len(imgs))], imgs, port, what="side stream")
        assert int(total.cpu()) == sum(len(want(port, im)) for im in imgs)
    finally:
        c.close()


def test_end_to_end_region_decode(ctx, port):
    sizes = [(500, 300), (37, 21), (1920, 1080), (264, 136), (96, 64), (1032, 40), (64, 48), (300, 5)]
    imgs = [image(port, w, h, 3, 8) for (w, h) in sizes]
    streams, _, _ = run_mixed(ctx, imgs, 3)
    rw, rh = 33, 5
    rng = np.random.default_rng(4)
    origins = [(int(rng.integers(0, w - rw + 1)), int(rng.integers(0, h - rh + 1))) for (w, h) in sizes]
    offs = np.cumsum([0] + [(len(s) + 15) & ~15 for s in streams])
    buf = np.zeros(offs[-1] + 64, np.uint8)
    for o, s in zip(offs, streams):
        buf[o: o + len(s)] = np.frombuffer(s, np.uint8)
    px, status = ctx.decode_batch_region_mixed(dev(buf), dev(offs[:-1].astype(np.int64)),
                                               dev(np.array([len(s) for s in streams], np.int32)),
                                               dev(np.array(sizes, np.int32)), 3, dev(np.array(origins, np.int32)), rw, rh,
                                               1920, 1080, 1)
    px, status = px.cpu().numpy(), status.cpu().numpy()
    assert list(status) == [OK] * len(sizes)
    for k, s in enumerate(streams):
        x, y = origins[k]
        whole = port.decode(s, strict=False)
        assert (px[k] == whole[y: y + rh, x: x + rw]).all(), f"image {k}"
