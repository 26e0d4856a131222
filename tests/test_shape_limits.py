"""Encode and decode at the limits of the accepted shapes and batch sizes, against the oracle.

The accepted shapes (include/himg_cuda.h): 1..255 channels, fewer than 2^31 pixel bytes, at most 65 535 block rows and
a block row of at most 2^26 coefficient bytes (8 * ceil(w / 8) * nch <= 2^23).  Between the sizes of the other tests
and these limits lies the 32-bit index and bit-count arithmetic of the kernels; the cases here sit on the limits:
shapes whose lane-pair inverse tiles start one division step away from a block-row boundary, the tallest and widest
images, images of about 2^31 pixel bytes, batches past the 65 535 grid limit and buffers past 2^32 bytes.

In every GPU case the oracle is the checker: encoded bytes are equal, decode gives the oracle's accept / reject decision
in both flag modes and its pixels, and a decoded region equals the crop of the oracle's whole decode.  Every GPU case
has its own context and frees its tensors; its docstring gives its peak device memory (estimated from the buffers)."""
import gc

import numpy as np
import pytest

OK, REJECT, ERR_ARG, ERR_UNSUPPORTED = 0, 1, 2, 5
STRICT, LENIENT = 0, 1
SEG_LIMIT = 1 << 23  # 8 * ceil(w / 8) * nch


# ---------------------------------------------------------------------------------------------
# CPU: the acceptance envelope
# ---------------------------------------------------------------------------------------------
def _accepted(lib, w, h, nch):
    bound, lres, stride = lib.himgcu_encode_bound(w, h, nch), lib.himgcu_lres_size(w, h, nch), lib.himgcu_lres_stride(w, h, nch)
    assert (bound > 0) == (lres > 0) == (stride > 0), (w, h, nch)
    return bound > 0


@pytest.mark.parametrize("edge, past", [
    ((SEG_LIMIT, 8, 1), (SEG_LIMIT + 1, 8, 1)),                  # block-row width, gray
    ((SEG_LIMIT - 7, 8, 1), (SEG_LIMIT + 1, 1, 1)),              # (same block columns; one pixel row past)
    ((SEG_LIMIT // 2, 16, 2), (SEG_LIMIT // 2 + 1, 16, 2)),
    ((2796200, 8, 3), (2796201, 8, 3)),                          # 8 * ceil(w / 8) * 3 = 8 388 600 / 8 388 624
    ((SEG_LIMIT // 8, 64, 8), (SEG_LIMIT // 8 + 1, 64, 8)),
    ((8, 524280, 1), (8, 524281, 1)),                            # 65 535 block rows / 65 536
    ((16, 524273, 3), (16, 524281, 3)),
    ((42966, 49981, 1), (32768, 65536, 1)),                      # 2^31 - 2 pixel bytes / 2^31 (2^31 - 1 is prime)
    ((21483, 49981, 2), (16384, 65536, 2)),
    ((3, 3, 255), (3, 3, 256)),                                  # channels
    # w + 7 and h + 7 overflow an int here: the rounding to blocks must not wrap to a negative count
    ((8, 8, 1), (2147483647, 1, 1)),
    ((8, 8, 1), (1, 2147483647, 1)),
    ((8, 8, 1), (2147483640, 1, 1)),                             # (fewer than 2^31 pixel bytes, a 2^34-byte block row)
    ((8, 8, 1), (1, 2147483641, 1)),
])
def test_acceptance_envelope(edge, past):
    """encode_bound / lres_size / lres_stride are non-zero exactly for the accepted shapes: each limit at its edge and
    one step past it."""
    from himg_b200 import _native

    lib = _native.load()
    assert _accepted(lib, *edge), edge
    assert not _accepted(lib, *past), past


def test_pixel_limit_edges_are_what_they_claim():
    assert 42966 * 49981 == (1 << 31) - 2 and 21483 * 2 * 49981 == (1 << 31) - 2
    assert 8 * ((2796200 + 7) // 8) * 3 <= SEG_LIMIT < 8 * ((2796201 + 7) // 8) * 3
    assert (524280 + 7) // 8 == 65535 and (524281 + 7) // 8 == 65536


# ---------------------------------------------------------------------------------------------
# GPU helpers
# ---------------------------------------------------------------------------------------------
def _torch():
    return pytest.importorskip("torch")


@pytest.fixture
def ctx():
    torch = _torch()
    import himg_b200

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    c = himg_b200.Context(0)
    c.set_stream(torch.cuda.current_stream().cuda_stream)
    yield c
    c.close()
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def dev(a):
    torch = _torch()
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def assert_same(got, want, what):
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, f"{what}: shape {got.shape} vs {want.shape}"
    idx = np.flatnonzero(got.reshape(-1) != want.reshape(-1))
    assert idx.size == 0, f"{what}: {idx.size} diffs, first at {int(idx[0])}"


def oracle(port, img, q, multi_row=None):
    """(stream, strict decode, lenient decode) of the oracle.  For an image of several block rows the two modes make
    the same framing decision, so a stream the strict decoder accepts decodes to the same pixels leniently and the
    second (slow, on the largest images) oracle decode is skipped."""
    s = port.encode(img, q, True)
    strict = port.decode(s, strict=True)
    if multi_row is None:
        multi_row = img.shape[0] > 8
    lenient = strict if (multi_row and strict is not None) else port.decode(s, strict=False)
    return s, strict, lenient


def check_encode_decode(c, port, img, q, what, regions=()):
    """GPU encode == oracle bytes; GPU decode == oracle decode in both flag modes; each (x, y, w, h) region == the crop.
    Returns the oracle's (stream, strict, lenient)."""
    s, strict, lenient = oracle(port, img, q)
    got = c.encode(img, q, True)
    assert got == s, f"{what}: encode differs ({len(got)} vs {len(s)} bytes)"
    del got
    for flags, want in ((STRICT, strict), (LENIENT, lenient)):
        d = c.decode(s, flags)
        assert (d is None) == (want is None), f"{what} flags {flags}: accept/reject differs"
        if want is not None:
            assert_same(d, want, f"{what} flags {flags}")
        del d
        for (x, y, w, h) in regions:
            r = c.decode_region(s, x, y, w, h, flags)
            assert (r is None) == (want is None), f"{what} region {(x, y, w, h)} flags {flags}"
            if want is not None:
                assert_same(r, want[y: y + h, x: x + w], f"{what} region {(x, y, w, h)} flags {flags}")
    return s, strict, lenient


def pack(streams, index):
    """Device buffer holding the distinct streams once, and offsets / sizes of image k = streams[index[k]]."""
    offs = np.cumsum([0] + [(len(s) + 15) & ~15 for s in streams])
    buf = np.zeros(offs[-1] + 64, np.uint8)
    for o, s in zip(offs, streams):
        buf[o: o + len(s)] = np.frombuffer(s, np.uint8)
    index = np.asarray(index)
    return (dev(buf), dev(offs[:-1][index].astype(np.int64)),
            dev(np.array([len(s) for s in streams], np.int32)[index]))


def raises_code(code, fn, *a, **k):
    import himg_b200

    with pytest.raises(himg_b200.HimgError) as e:
        fn(*a, **k)
    assert e.value.code == code, str(e.value)


def small_out(n=1):
    """Output rows for a batch encode of a shape without an encode bound (the call must refuse the shape itself)."""
    torch = _torch()
    return dict(out=torch.empty((n, 256), dtype=torch.uint8, device="cuda"), sizes=torch.empty(n, dtype=torch.int32, device="cuda"))


def patch_height(s, h):
    """The stream with its FRMT height replaced (RIFF header 12 bytes, chunk header 8, version 1, width 4)."""
    b = bytearray(s)
    assert b[12:16] == b"FRMT"
    b[25:29] = int(h).to_bytes(4, "little")
    return bytes(b)


def patch_width(s, w):
    b = bytearray(s)
    assert b[12:16] == b"FRMT"
    b[21:25] = int(w).to_bytes(4, "little")
    return bytes(b)


# ---------------------------------------------------------------------------------------------
# 1. Lane-pair inverse: shapes whose tile starts lie just below a block-row boundary
# ---------------------------------------------------------------------------------------------
# A CTA of the lane-pair inverse owns 256 consecutive block pairs; its first block row is f0 / PR (PR = pairs per
# block row).  On these shapes a 32-bit reciprocal of PR is one too large for some tile: 3088512 x 8 (last tile),
# 106368 x 6648 (last tile) and 1811840 x 24 x 3 (last tile) one row past the image, 68480 x 17120 six tiles one row
# too far down.  The whole-image decode and decode_batch run that kernel (k_inverse4); decode_region runs
# k_inverse_region4, which divides, so the regions here check the crop path on these shapes, not the quotient.
@pytest.mark.gpu
def test_inverse_tile_rows_thin_gray(ctx, port):
    """3088512 x 8 gray (24.7 MP): stage_inverse on random planes, encode / decode, a two-image decode_batch (a tile read
    past image 0 would land in image 1) and a bottom-right region.  Peak device memory about 0.5 GB."""
    torch = _torch()
    w, h = 3088512, 8
    rng = np.random.default_rng(5)
    cols = w // 8
    planes = rng.choice(np.array([0, 0, 0, 1, 255, 2, 254, 9, 247], np.uint8), cols * 64)
    R = rng.integers(0, 256, (1, 1, cols), dtype=np.uint8)
    unmap = port.mapfun_parse(port.mapfun_serialize(port.fullres_map_table()))
    sl, sc = port.shift_table(50, 0), port.shift_table(50, 1)
    want = port.fullres_restore(planes, w, h, 1, False, R, sl, sc, unmap)
    got = ctx.stage_inverse(dev(planes[None]), dev(R[None]), w, h, 1, False, sl, sc, unmap).cpu().numpy()[0]
    assert_same(got, want, "stage_inverse")
    del got, want

    imgs = [port.synth(w, h, 1, seed, 6) for seed in (3, 4)]
    wants = [check_encode_decode(ctx, port, imgs[0], 50, "thin gray", regions=[(w - 224, 0, 224, 8), (w - 37, 3, 37, 5)])]
    wants.append(oracle(port, imgs[1], 50))
    himg, offs, sizes = pack([x[0] for x in wants], [0, 1])
    for flags in (STRICT, LENIENT):
        out, status = ctx.decode_batch(himg, offs, sizes, w, h, 1, flags)
        out, status = out.cpu().numpy(), status.cpu().numpy()
        for k in range(2):
            want = wants[k][1 + flags]
            assert status[k] == (OK if want is not None else REJECT), (flags, k)
            if want is not None:
                assert_same(out[k], want, f"decode_batch image {k} flags {flags}")
    del out, himg
    torch.cuda.synchronize()


@pytest.mark.gpu
@pytest.mark.parametrize("w, h, nch, region", [
    (106368, 6648, 1, (106368 - 224, 6648 - 224, 224, 224)),
    (1811840, 24, 3, (1811840 - 224, 0, 224, 24)),
    # the tile at pair 8 384 512 starts 8 pairs before the end of block row 1958 and runs into row 1959
    (68480, 17120, 1, (68480 - 256, 8 * 1958, 256, 16)),
])
def test_inverse_tile_rows(ctx, port, w, h, nch, region):
    """Encode / decode of the shapes the reciprocal misplaced (the decode is the check of k_inverse4), and a region over
    the misplaced tile (the region kernel's crop of the same pixels).  Peak device memory
    about 6 x the pixel bytes: 4.2 GB for 106368 x 6648, 4 GB for 1811840 x 24 x 3, 7 GB for 68480 x 17120."""
    img = port.synth(w, h, nch, 7, 6)
    x, y, rw, rh = region
    check_encode_decode(ctx, port, img, 50, f"{w}x{h}x{nch}", regions=[region, (x + rw - 16, y + rh - 8, 16, 8)])


# ---------------------------------------------------------------------------------------------
# 2. Tallest images: 65 535 block rows
# ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("nch", [1, 3])
@pytest.mark.parametrize("w", [8, 13, 16])
def test_tallest_images(ctx, port, w, nch):
    """h = 524 280 (65 535 block rows): encode, decode, the last 8 rows as a region, and the image in a mixed batch
    next to small images; h = 524 281 is ERR_UNSUPPORTED from encode, encode_batch and the decode of a stream whose
    FRMT height is patched to it.  Peak device memory about 1 GB."""
    torch = _torch()
    h = 524280
    img = port.synth(w, h, nch, 11, 6)
    tall = check_encode_decode(ctx, port, img, 50, f"tall {w}x{nch}", regions=[(0, h - 8, w, 8), (w - 1, h - 3, 1, 3)])

    # mixed batch: the tall image between small ones
    small = [port.synth(sw, sh, nch, 12, 6) for sw, sh in ((16, 40), (3, 5), (13, 8))]
    imgs = [small[0], img, small[1], small[2]]
    wants = [oracle(port, small[0], 50), tall, oracle(port, small[1], 50), oracle(port, small[2], 50)]
    dims = np.array([(im.shape[1], im.shape[0]) for im in imgs], np.int32)
    offs = np.cumsum([0] + [im.size for im in imgs])
    flat = np.concatenate([im.reshape(-1) for im in imgs])
    out, sizes = ctx.encode_batch_mixed(dev(flat), dev(offs[:-1].astype(np.int64)), dev(dims), nch, 16, h)
    rows, sizes = out.cpu().numpy(), sizes.cpu().numpy()
    for k, want in enumerate(wants):
        assert rows[k, : sizes[k]].tobytes() == want[0], f"encode_batch_mixed image {k}"
    del out, rows
    himg, o, sz = pack([x[0] for x in wants], range(4))
    for flags in (STRICT, LENIENT):
        px, poff, status = ctx.decode_batch_mixed(himg, o, sz, dev(dims), nch, 16, h, flags)
        px, poff, status = px.cpu().numpy(), poff.cpu().numpy(), status.cpu().numpy()
        for k, want in enumerate(wants):
            want = want[1 + flags]
            assert status[k] == (OK if want is not None else REJECT), (flags, k)
            if want is not None:
                assert_same(px[poff[k]: poff[k] + want.size].reshape(want.shape), want, f"decode_batch_mixed {k} flags {flags}")
        del px

    # one pixel row more is one block row too many
    big = np.zeros((h + 1, w, nch), np.uint8)
    raises_code(ERR_UNSUPPORTED, ctx.encode, big, 50)
    raises_code(ERR_UNSUPPORTED, ctx.encode_batch, dev(big[None]), **small_out())
    for flags in (STRICT, LENIENT):
        raises_code(ERR_UNSUPPORTED, ctx.decode, patch_height(tall[0], h + 1), flags)
    del big
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------
# 3. Widest block rows: 8 * ceil(w / 8) * nch = 2^23
# ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("content", ["noise-q100", "synth-q50"])
@pytest.mark.parametrize("h", [8, 13])
@pytest.mark.parametrize("nch", [1, 3])
def test_widest_block_rows(ctx, port, nch, h, content):
    """The widest accepted block row (2^26 coefficient bytes): random noise at q100 gives the largest coded rows (one
    unframed segment at h = 8), the synthetic image at q50 the usual ones.  Peak device memory about 2 GB."""
    w = SEG_LIMIT // nch - (SEG_LIMIT // nch) % 8
    if content == "noise-q100":
        img, q = np.random.default_rng(h + nch).integers(0, 256, (h, w, nch), dtype=np.uint8), 100
    else:
        img, q = port.synth(w, h, nch, 13, 6), 50
    check_encode_decode(ctx, port, img, q, f"wide {w}x{h}x{nch} {content}", regions=[(w - 224, h - 8, 224, 8)])


@pytest.mark.gpu
@pytest.mark.parametrize("nch", [1, 3])
def test_one_step_past_the_widest_block_row(ctx, port, nch):
    """A block row one block column past 2^26 bytes is ERR_UNSUPPORTED from every entry point: encode, both batch
    encodes (as a shape and as mixed bounds), every batch decode, and decode / decode_region of a stream whose FRMT
    width is patched to it.  Peak device memory about 0.3 GB."""
    torch = _torch()
    w = SEG_LIMIT // nch - (SEG_LIMIT // nch) % 8 + 8
    img = np.zeros((8, w, nch), np.uint8)
    raises_code(ERR_UNSUPPORTED, ctx.encode, img, 50)
    raises_code(ERR_UNSUPPORTED, ctx.encode_batch, dev(img[None]), **small_out())
    small = port.synth(16, 8, nch, 1, 6)
    s = port.encode(small, 50, True)
    dims = dev(np.array([[16, 8]], np.int32))
    raises_code(ERR_UNSUPPORTED, ctx.encode_batch_mixed, dev(small.reshape(-1)), dev(np.zeros(1, np.int64)), dims, nch, w, 8,
                **small_out())
    himg, offs, sizes = pack([s], [0])
    origins = dev(np.zeros((1, 2), np.int32))
    raises_code(ERR_UNSUPPORTED, ctx.decode_batch, himg, offs, sizes, w, 8, nch)
    raises_code(ERR_UNSUPPORTED, ctx.decode_batch_region, himg, offs, sizes, w, 8, nch, origins, 8, 8)
    out = torch.empty(16 * 8 * nch, dtype=torch.uint8, device="cuda")
    raises_code(ERR_UNSUPPORTED, ctx.decode_batch_mixed, himg, offs, sizes, dims, nch, w, 8, out=out,
                pixel_offsets=dev(np.zeros(1, np.int64)))
    raises_code(ERR_UNSUPPORTED, ctx.decode_batch_region_mixed, himg, offs, sizes, dims, nch, origins, 8, 8, w, 8)
    bad = patch_width(s, w)
    for flags in (STRICT, LENIENT):
        raises_code(ERR_UNSUPPORTED, ctx.decode, bad, flags)
        raises_code(ERR_UNSUPPORTED, ctx.decode_region, bad, 0, 0, 8, 8, flags)
    # the edge itself is accepted as mixed bounds
    out, sz = ctx.encode_batch_mixed(dev(small.reshape(-1)), dev(np.zeros(1, np.int64)), dims, nch, w - 8, 8)
    assert out[0, : int(sz[0])].cpu().numpy().tobytes() == s


# ---------------------------------------------------------------------------------------------
# 4. About 2^31 pixel bytes
# ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("w, h, nch", [
    (26753, 26753, 3),  # padded to 26760^2: 2 148 292 800 plane bytes (> 2^31), the generic kernels
    (46336, 46336, 1),  # the lane-pair kernels, 2 147 024 896 plane bytes in one launch
])
def test_near_the_pixel_limit(ctx, port, w, h, nch):
    """q50: encode bytes, decode pixels in both modes, a 224^2 region at the bottom-right.  Peak device memory about
    8 x the pixel bytes, 17 GB."""
    assert w * h * nch < (1 << 31)
    img = port.synth(w, h, nch, 17, 6)
    check_encode_decode(ctx, port, img, 50, f"{w}x{h}x{nch}", regions=[(w - 224, h - 224, 224, 224)])


# ---------------------------------------------------------------------------------------------
# 5. Batches past the 65 535 grid limit
# ---------------------------------------------------------------------------------------------
NBIG = 65544
SMALL = [(8, 8), (1, 1), (17, 3)]


def _check_rows(rows, sizes, index, streams, what):
    for j, s in enumerate(streams):
        sel = np.flatnonzero(index == j)
        assert (sizes[sel] == len(s)).all(), f"{what}: sizes of stream {j}"
        want = np.frombuffer(s, np.uint8)
        bad = np.flatnonzero((rows[sel, : len(s)] != want).any(axis=1))
        assert bad.size == 0, f"{what}: image {int(sel[bad[0]])} differs"


def _check_images(px, status, index, wants, what):
    """px [n][...] against wants[index[k]] (None: REJECT; an int: that status, pixels not written)."""
    for j, want in enumerate(wants):
        sel = np.flatnonzero(index == j)
        code = want if isinstance(want, int) else OK if want is not None else REJECT
        assert (status[sel] == code).all(), f"{what}: status of image kind {j}"
        if code == OK:
            bad = np.flatnonzero((px[sel].reshape(sel.size, -1) != want.reshape(-1)).any(axis=1))
            assert bad.size == 0, f"{what}: image {int(sel[bad[0]])} differs"


@pytest.mark.gpu
@pytest.mark.parametrize("w, h", SMALL)
def test_batches_past_the_grid_limit(ctx, port, w, h):
    """n = 65 544 images of one small shape, image k = seed k % 4, through encode_batch, decode_batch and
    decode_batch_region; every image is checked.  Peak device memory about 0.5 GB."""
    nch = 3
    index = np.arange(NBIG) % 4
    imgs = [port.synth(w, h, nch, 20 + j, 6) for j in range(4)]
    wants = [oracle(port, im, 50) for im in imgs]
    out, sizes = ctx.encode_batch(dev(np.stack(imgs)[index]), 50, True)
    _check_rows(out.cpu().numpy(), sizes.cpu().numpy(), index, [x[0] for x in wants], "encode_batch")
    del out
    himg, offs, sz = pack([x[0] for x in wants], index)
    cw, ch = max(1, w // 2), max(1, h // 2)
    ox, oy = w - cw, h - ch
    origins = dev(np.tile(np.array([ox, oy], np.int32), (NBIG, 1)))
    for flags in (STRICT, LENIENT):
        px, status = ctx.decode_batch(himg, offs, sz, w, h, nch, flags)
        _check_images(px.cpu().numpy(), status.cpu().numpy(), index, [x[1 + flags] for x in wants], f"decode_batch {flags}")
        px, status = ctx.decode_batch_region(himg, offs, sz, w, h, nch, origins, cw, ch, flags)
        crops = [None if x[1 + flags] is None else x[1 + flags][oy: oy + ch, ox: ox + cw] for x in wants]
        _check_images(px.cpu().numpy(), status.cpu().numpy(), index, crops, f"decode_batch_region {flags}")
    del px


@pytest.mark.gpu
def test_mixed_batches_past_the_grid_limit(ctx, port):
    """n = 65 544 images cycling through 8x8, 1x1 and 17x3 (four seeds each) through encode_batch_mixed,
    decode_batch_mixed and decode_batch_region_mixed; every image is checked.  Peak device memory about 1 GB."""
    torch = _torch()
    nch = 3
    kinds = [(w, h, seed) for (w, h) in SMALL for seed in range(4)]
    index = np.arange(NBIG) % len(kinds)
    imgs = [port.synth(w, h, nch, 30 + seed, 6) for (w, h, seed) in kinds]
    wants = [oracle(port, im, 50) for im in imgs]
    dims_k = np.array([(w, h) for (w, h, _) in kinds], np.int32)
    dims = dev(dims_k[index])
    spans = np.array([im.size for im in imgs])[index]
    offs = np.cumsum(np.concatenate([[0], spans]))
    flat = np.concatenate([imgs[j].reshape(-1) for j in index])
    out, sizes = ctx.encode_batch_mixed(dev(flat), dev(offs[:-1].astype(np.int64)), dims, nch, 17, 8)
    _check_rows(out.cpu().numpy(), sizes.cpu().numpy(), index, [x[0] for x in wants], "encode_batch_mixed")
    del out
    himg, o, sz = pack([x[0] for x in wants], index)
    # regions: the bottom-right pixel of every image, and an 8 x 3 rectangle at the bottom-right of the images it fits
    # (ERR_ARG for the 1 x 1 images)
    corner = dev((dims_k - 1)[index])
    rect = dev(np.maximum(dims_k - np.array([8, 3], np.int32), 0)[index])
    for flags in (STRICT, LENIENT):
        px, poff, status = ctx.decode_batch_mixed(himg, o, sz, dims, nch, 17, 8, flags)
        px, poff, status = px.cpu().numpy(), poff.cpu().numpy(), status.cpu().numpy()
        assert (poff == offs[:-1]).all()
        for j, x in enumerate(wants):
            want = x[1 + flags]
            sel = np.flatnonzero(index == j)
            assert (status[sel] == (OK if want is not None else REJECT)).all(), f"decode_batch_mixed {flags} kind {j}"
            if want is not None:
                got = px[poff[sel][:, None] + np.arange(want.size)[None, :]]
                bad = np.flatnonzero((got != want.reshape(-1)).any(axis=1))
                assert bad.size == 0, f"decode_batch_mixed {flags}: image {int(sel[bad[0]])} differs"
        del px
        px, status = ctx.decode_batch_region_mixed(himg, o, sz, dims, nch, corner, 1, 1, 17, 8, flags)
        crops = [None if x[1 + flags] is None else x[1 + flags][-1:, -1:] for x in wants]
        _check_images(px.cpu().numpy(), status.cpu().numpy(), index, crops, f"decode_batch_region_mixed 1x1 {flags}")
        px, status = ctx.decode_batch_region_mixed(himg, o, sz, dims, nch, rect, 8, 3, 17, 8, flags)
        crops = [ERR_ARG if w < 8 else None if x[1 + flags] is None else x[1 + flags][-3:, -8:]
                 for (w, _, _), x in zip(kinds, wants)]
        _check_images(px.cpu().numpy(), status.cpu().numpy(), index, crops, f"decode_batch_region_mixed 8x3 {flags}")
        del px
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------
# 6. Buffers past 2^32 bytes
# ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_batch_buffers_past_4_gib(ctx, port):
    """700 x 1080p RGB (4.35 GB of pixels, image k = synth seed k % 4) through encode_batch and decode_batch in both flag
    modes; all 700 are checked against the four oracle results.  Peak device memory about 25 GB."""
    torch = _torch()
    from himg_b200.synth import synth_images

    n, w, h, nch = 700, 1920, 1080, 3
    base = synth_images(4, w, h, nch, 40, 6)
    index = torch.arange(n, device="cuda") % 4
    wants = [oracle(port, base[j].cpu().numpy(), 50) for j in range(4)]
    pixels = base[index]
    out, sizes = ctx.encode_batch(pixels, 50, True)
    del pixels
    sizes = sizes.cpu().numpy()
    for j, (s, _, _) in enumerate(wants):
        assert (sizes[j::4] == len(s)).all(), f"encode_batch sizes of seed {j}"
        assert bool((out[j::4, : len(s)] == dev(np.frombuffer(s, np.uint8))[None]).all()), f"encode_batch seed {j}"
    del out
    himg, offs, sz = pack([x[0] for x in wants], np.arange(n) % 4)
    for flags in (STRICT, LENIENT):
        px, status = ctx.decode_batch(himg, offs, sz, w, h, nch, flags)
        status = status.cpu().numpy()
        for j, x in enumerate(wants):
            want = x[1 + flags]
            assert want is not None and (status[j::4] == OK).all(), f"decode_batch seed {j} flags {flags}"
            assert bool((px[j::4] == dev(want)[None]).all()), f"decode_batch seed {j} flags {flags}"
        del px
    del base
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_mixed_workspace_and_pixel_offsets_past_4_gib(ctx, port):
    """24 small images under 8192 x 8192 x 3 bounds (workspace slots of the later images lie past 4 GiB), with the
    caller's pixel offsets of both mixed calls past 2^32.  Peak device memory about 30 GB."""
    torch = _torch()
    nch, mw, mh, base_off = 3, 8192, 8192, (1 << 32) + 77
    shapes = [(64, 48), (1, 1), (17, 3), (500, 300), (1920, 1080), (40, 8)] * 4
    imgs = [port.synth(w, h, nch, 50 + k, 6) for k, (w, h) in enumerate(shapes)]
    wants = [oracle(port, im, 50) for im in imgs]
    dims = dev(np.array(shapes, np.int32))
    spans = np.array([im.size for im in imgs])
    offs = base_off + np.cumsum(np.concatenate([[0], spans + 5]))[:-1]
    pixels = torch.zeros(int(offs[-1] + spans[-1] + 64), dtype=torch.uint8, device="cuda")
    for o, im in zip(offs, imgs):
        pixels[int(o): int(o) + im.size] = dev(im.reshape(-1))
    out, sizes = ctx.encode_batch_mixed(pixels, dev(offs.astype(np.int64)), dims, nch, mw, mh)
    sizes = sizes.cpu().numpy()
    for k, (s, _, _) in enumerate(wants):
        assert out[k, : sizes[k]].cpu().numpy().tobytes() == s, f"encode_batch_mixed image {k} {shapes[k]}"
    del out
    himg, o, sz = pack([x[0] for x in wants], range(len(wants)))
    for flags in (STRICT, LENIENT):
        pixels.fill_(0xA5)
        _, _, status = ctx.decode_batch_mixed(himg, o, sz, dims, nch, mw, mh, flags, out=pixels,
                                              pixel_offsets=dev(offs.astype(np.int64)))
        status = status.cpu().numpy()
        for k, x in enumerate(wants):
            want = x[1 + flags]
            assert status[k] == (OK if want is not None else REJECT), (flags, k)
            if want is not None:
                got = pixels[int(offs[k]): int(offs[k]) + want.size].cpu().numpy()
                assert_same(got.reshape(want.shape), want, f"decode_batch_mixed image {k} {shapes[k]} flags {flags}")
        assert int((pixels[: int(offs[0])] != 0xA5).sum()) == 0, "a byte before the first span was written"
    del pixels
    torch.cuda.synchronize()
