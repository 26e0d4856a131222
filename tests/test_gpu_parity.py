"""GPU parity tests: the CUDA path (through the C ABI) against the oracle, bit for bit.

Every test calls libhimgcu.so through himg_b200 (ctypes); the oracle is only the checker.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


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


def first_diff(a, b):
    a = np.asarray(a).reshape(-1)
    b = np.asarray(b).reshape(-1)
    if a.size != b.size:
        return f"size {a.size} vs {b.size}"
    idx = np.flatnonzero(a != b)
    if idx.size == 0:
        return None
    i = int(idx[0])
    return f"{idx.size} diffs, first at {i}: got {a[max(0, i - 4): i + 8].tolist()} want {b[max(0, i - 4): i + 8].tolist()}"


def assert_same(got, want, what):
    d = first_diff(got, want)
    assert d is None, f"{what}: {d}"


def rand_image(rng, w, h, n, kind):
    if kind == 0:
        yy, xx = np.mgrid[0:h, 0:w]
        img = np.stack([(xx * 2 + yy + 40 * c) % 256 for c in range(n)], -1)
        return (img + rng.integers(-60, 61, img.shape)).clip(0, 255).astype(np.uint8)
    if kind == 1:
        return np.full((h, w, n), int(rng.integers(0, 256)), np.uint8)
    if kind == 2:
        return rng.integers(0, 256, (h, w, n), dtype=np.uint8)
    img = np.zeros((h, w, n), np.uint8)
    img[rng.random((h, w)) < 0.02] = 255
    return img


SHAPES = [(64, 48, 3), (40, 24, 1), (37, 21, 1), (96, 64, 4), (500, 300, 3), (512, 300, 3), (8, 8, 1), (1, 1, 3),
          (1032, 40, 3), (2056, 16, 1), (136, 264, 2), (264, 136, 4)]


FLAT_SHAPES = [(1920, 64, 3), (272, 200, 3), (16, 4104, 1), (4112, 16, 3), (3840, 24, 3), (1040, 72, 1), (304, 136, 4),
               (32, 2072, 3)]


# ---------------------------------------------------------------------------------------------
# stages, encode side
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("ycbcr", [True, False])
def test_stage_lowres(ctx, port, shape, ycbcr):
    w, h, n = shape
    img = port.synth(w, h, n, 5, 9)
    yc = ycbcr and n >= 3
    cm = port.rgb_to_ycbcr(img) if yc else img
    want = port.lowres_sample(cm)
    got = ctx.stage_lowres(dev(img[None]), yc).cpu().numpy()[0]
    assert_same(got, want, f"lowres {shape} ycbcr={yc}")


def test_stage_lowres_lane_pair_path(ctx, port):
    # width % 16 == 0: k_lowres_avg2 (block pairs, dp4a colour map) for 1, 3 and 4 channels, more than
    # one CTA per window row (4112 / 16 > 128 pairs), single block rows and clipped top / bottom windows
    for (w, h, n) in FLAT_SHAPES + [(16, 8, 3), (48, 13, 1)]:
        for ycbcr in (True, False):
            img = port.synth(w, h, n, 11, 40)
            yc = ycbcr and n >= 3
            cm = port.rgb_to_ycbcr(img) if yc else img
            got = ctx.stage_lowres(dev(np.stack([img, img[:, ::-1].copy()])), yc).cpu().numpy()
            assert_same(got[0], port.lowres_sample(cm), f"lowres {(w, h, n)} ycbcr={yc}")
            cm1 = port.rgb_to_ycbcr(img[:, ::-1].copy()) if yc else img[:, ::-1].copy()
            assert_same(got[1], port.lowres_sample(cm1), f"lowres, second image {(w, h, n)}")


def test_stage_lowres_batch_and_stride(ctx, port):
    rng = np.random.default_rng(1)
    imgs = np.stack([rand_image(rng, 200, 120, 3, k % 4) for k in range(5)])
    got = ctx.stage_lowres(dev(imgs), True).cpu().numpy()
    for k in range(5):
        assert_same(got[k], port.lowres_sample(port.rgb_to_ycbcr(imgs[k])), f"image {k}")
    # 3 channels out of 4-byte pixels (pixel_stride > num_channels)
    img4 = rand_image(rng, 72, 40, 4, 0)
    got = ctx.stage_lowres(dev(img4[None]), True, nch=3).cpu().numpy()[0]
    assert_same(got, port.lowres_sample(port.rgb_to_ycbcr(np.ascontiguousarray(img4[:, :, :3]))), "stride 4")


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("quality", [0, 50, 100])
def test_stage_lres_encode(ctx, port, shape, quality):
    w, h, n = shape
    img = port.synth(w, h, n, 6, 12)
    L = port.lowres_sample(img)
    want = port.lowres_encode(L, quality)
    out, size = ctx.stage_lres_encode(dev(L[None]), w, h, quality)
    assert size == want.size
    assert_same(out.cpu().numpy()[0, :size], want, f"lres {shape} q{quality}")


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("quality,ycbcr", [(50, True), (0, True), (100, True), (77, False)])
def test_stage_forward(ctx, port, shape, quality, ycbcr):
    w, h, n = shape
    img = port.synth(w, h, n, 7, 20)
    yc = ycbcr and n >= 3
    cm = port.rgb_to_ycbcr(img) if yc else img
    L = port.lowres_sample(cm)
    want = port.fullres_planes(cm, L, quality, yc)
    got = ctx.stage_forward(dev(img[None]), dev(L[None]), quality, yc).cpu().numpy()[0]
    assert_same(got, want, f"planes {shape} q{quality} ycbcr={yc}")


# Flat tiles (256 consecutive block pairs per CTA, whatever the width): tiles that start and end inside
# a block row, many block rows per tile (more than the 32 lanes that issue the bulk copies), rows wider
# than a tile, a last tile with idle threads.


@pytest.mark.parametrize("shape", FLAT_SHAPES)
@pytest.mark.parametrize("quality,ycbcr", [(50, True), (100, True), (33, False)])
def test_stage_forward_flat_tiles(ctx, port, shape, quality, ycbcr):
    w, h, n = shape
    img = port.synth(w, h, n, 17, 25)
    yc = ycbcr and n >= 3
    cm = port.rgb_to_ycbcr(img) if yc else img
    L = port.lowres_sample(cm)
    want = port.fullres_planes(cm, L, quality, yc)
    got = ctx.stage_forward(dev(np.stack([img, img[::-1].copy()])), dev(np.stack([L, L])), quality, yc).cpu().numpy()
    assert_same(got[0], want, f"planes {shape} q{quality} ycbcr={yc}")
    cm1 = port.rgb_to_ycbcr(img[::-1].copy()) if yc else img[::-1].copy()
    assert_same(got[1], port.fullres_planes(cm1, L, quality, yc), f"second image {shape}")


def test_stage_forward_extreme_values(ctx, port):
    """Checkerboards drive |T| to its 16320 maximum and exercise the top of MapTo8Bit."""
    yy, xx = np.mgrid[0:64, 0:128]
    for pat in (((xx + yy) & 1) * 255, (xx & 1) * 255, ((xx >> 2) & 1) * 255, ((yy >> 1) & 1) * 255):
        img = np.repeat(pat[:, :, None], 3, 2).astype(np.uint8)
        for q in (100, 50):
            L = port.lowres_sample(img)
            want = port.fullres_planes(img, L, q, False)
            got = ctx.stage_forward(dev(img[None]), dev(L[None]), q, False).cpu().numpy()[0]
            assert_same(got, want, f"extreme q{q}")


def _huff_cases():
    rng = np.random.default_rng(11)
    cases = []
    for trial in range(12):
        nseg = [1, 1, 2, 3, 8, 5, 1, 4, 16, 2, 1, 7][trial]
        seg = [1, 100, 64, 3000, 512, 20000, 70000, 46080, 4096, 40000, 16384 * 3, 33][trial]
        n = nseg * seg
        data = rng.integers(0, 256, n, dtype=np.uint8)
        data[rng.random(n) < [0.0, 0.5, 0.9, 0.99, 0.7, 0.95, 0.999, 0.8, 0.3, 1.0, 0.97, 0.6][trial]] = 0
        if trial % 4 == 1:
            data = (data % 5).astype(np.uint8)
        cases.append((data, 0 if nseg == 1 else seg))
    z = np.zeros(60000, np.uint8)  # runs longer than 16662, cut greedily
    z[[19999, 39998]] = 5
    cases += [(z, 0), (z, 20000), (np.zeros(50000, np.uint8), 0), (np.zeros(50000, np.uint8), 10000),
              (np.full(5000, 7, np.uint8), 0), (np.full(5000, 7, np.uint8), 1000)]
    # Fibonacci symbol counts 1, 1, 2, 3, 5, ... over {literal 24, run symbol 260, run symbol 259, literals
    # 23 .. 1}: codes of up to 26 bits.  "5000 zeros + literal 24" is one item of 40 + 26 bits (> 64),
    # "100 zeros + literal 23" one of 33 + 24 bits (> 32): the wide-item paths of the packer and the
    # tree walk of the decoder.
    f = [1, 1]
    while len(f) < 27:
        f.append(f[-1] + f[-2])
    dense = np.concatenate([np.full(f[26 - k] - (2 if k == 22 else 0), k + 1, np.uint8) for k in range(23)])  # literals 1..23
    rng.shuffle(dense)
    z = lambda n, v: np.r_[np.zeros(n, np.uint8), np.uint8(v)]
    deep = np.concatenate([dense[:1000], [np.uint8(25)], dense[1000:70001], z(5000, 24), dense[70001:300000], z(100, 23), dense[300000:300007], z(200, 23),
                           dense[300007:]])
    deep = deep[: deep.size & ~3]
    cases += [(deep, 0)]
    return cases


def test_stage_huff_compress(ctx, port):
    for k, (data, bs) in enumerate(_huff_cases()):
        want = port.huff_compress(data, bs)
        out, sizes = ctx.stage_huff_compress(dev(data[None]), bs)
        ctx.encode_status()
        size = int(sizes.cpu()[0])
        assert size == len(want), f"case {k}: size {size} vs {len(want)}"
        assert_same(out.cpu().numpy()[0, :size], np.frombuffer(want, np.uint8), f"huff case {k} (n={data.size}, bs={bs})")


def test_stage_huff_compress_batch(ctx, port):
    rng = np.random.default_rng(12)
    data = rng.integers(0, 256, (6, 8 * 2048), dtype=np.uint8)
    for i in range(6):
        data[i][rng.random(data.shape[1]) < 0.15 * i] = 0
    out, sizes = ctx.stage_huff_compress(dev(data), 2048)
    ctx.encode_status()
    out, sizes = out.cpu().numpy(), sizes.cpu().numpy()
    for i in range(6):
        want = port.huff_compress(data[i], 2048)
        assert sizes[i] == len(want)
        assert_same(out[i, : sizes[i]], np.frombuffer(want, np.uint8), f"item {i}")


# ---------------------------------------------------------------------------------------------
# whole encoder
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("quality,ycbcr", [(50, True), (5, True), (100, True), (60, False)])
def test_encode_matches_oracle(ctx, port, shape, quality, ycbcr):
    w, h, n = shape
    img = port.synth(w, h, n, 3, 6)
    got = ctx.encode(img, quality, ycbcr)
    want = port.encode(img, quality, ycbcr)
    assert len(got) == len(want), f"size {len(got)} vs {len(want)}"
    assert_same(np.frombuffer(got, np.uint8), np.frombuffer(want, np.uint8), f"himg {shape} q{quality}")


def test_encode_fixture_bitstreams(ctx, port, fixtures):
    i = 0
    while f"case{i}_meta" in fixtures:
        w, h, n, q, seed, amp, yc = (int(x) for x in fixtures[f"case{i}_meta"])
        got = ctx.encode(port.synth(w, h, n, seed, amp), q, bool(yc))
        assert_same(np.frombuffer(got, np.uint8), fixtures[f"case{i}_himg"], f"fixture {i}")
        i += 1


def test_encode_random_content(ctx, port):
    rng = np.random.default_rng(21)
    for k, (w, h, n) in enumerate([(256, 128, 3), (128, 256, 1), (320, 200, 4), (72, 72, 3)]):
        for kind in range(4):
            for q in (20, 50, 90, 100):
                img = rand_image(rng, w, h, n, kind)
                got, want = ctx.encode(img, q, True), port.encode(img, q, True)
                assert_same(np.frombuffer(got, np.uint8), np.frombuffer(want, np.uint8), f"{w}x{h}x{n} kind{kind} q{q}")


def test_encode_pixel_stride(ctx, port):
    rng = np.random.default_rng(5)
    img = rand_image(rng, 56, 40, 4, 0)
    got = ctx.encode(img, 50, True, pixel_stride=4, w=56, h=40, nch=3)
    assert got == port.encode(np.ascontiguousarray(img[:, :, :3]), 50, True)


def _golden(golden_hashes, w, h, n, q, seed=1):
    for c in golden_hashes:
        if (c["w"], c["h"], c["nch"], c["quality"], c["seed"], c["amp"], c["ycbcr"]) == (w, h, n, q, seed, 6, 1):
            return c
    raise KeyError((w, h, n, q))


@pytest.mark.parametrize("cfg", [(512, 512, 3, 50), (3840, 2160, 3, 50), (8192, 8192, 1, 50), (8192, 16, 1, 100)] +
                         [(1920, 1080, 3, q) for q in range(0, 101, 10)])  # c1, c2, c3, 4-byte headers, c4/c5 sweep
def test_golden_configs_encode_decode(ctx, port, golden_hashes, cfg):
    """BASELINE.json configurations at full size against the reference's recorded hashes."""
    w, h, n, q = cfg
    c = _golden(golden_hashes, w, h, n, q, 7 if (w, h) == (8192, 16) else 1)
    img = port.synth(w, h, n, c["seed"], c["amp"])
    packed = ctx.encode(img, q, True)
    assert len(packed) == c["himg_size"]
    assert f"{port.fnv(np.frombuffer(packed, np.uint8)):016x}" == c["himg_hash"]
    dec = ctx.decode(packed)
    if c["ref_decode"] == "fails":
        assert dec is None
        assert ctx.decode(packed, flags=1) is not None
    else:
        assert dec is not None
        assert f"{port.fnv(dec):016x}" == c["pixel_hash"]


# ---------------------------------------------------------------------------------------------
# stages, decode side
# ---------------------------------------------------------------------------------------------
def test_stage_huff_uncompress(ctx, port):
    for k, (data, bs) in enumerate(_huff_cases()):
        if data.size % 4 or (bs and bs % 4):
            continue
        packed = np.frombuffer(port.huff_compress(data, bs), np.uint8)
        buf = np.zeros((1, (packed.size + 67) & ~63), np.uint8)
        buf[0, : packed.size] = packed
        sizes = dev(np.array([packed.size], np.int32))
        for flags in (0, 1):
            out, status = ctx.stage_huff_uncompress(dev(buf), sizes, data.size, bs, flags)
            nseg = 1 if not bs else data.size // bs
            want_ok = True
            if bs:
                want_ok = all(port.huff_uncompress(packed.tobytes(), bs, bs, b, strict=(flags == 0), unpacked_total=data.size) is not None for b in range(nseg))
            else:
                want_ok = port.huff_uncompress(packed.tobytes(), data.size, 0, -1, strict=(flags == 0), unpacked_total=data.size) is not None
            got_ok = int(status.cpu()[0]) == 0
            assert got_ok == want_ok, f"case {k} flags {flags}: status {got_ok} vs oracle {want_ok}"
            if want_ok:
                assert_same(out.cpu().numpy()[0], data, f"uncompress case {k} flags {flags}")


def test_stage_lres_decode(ctx, port):
    for (w, h, n) in SHAPES:
        for q in (0, 50):
            img = port.synth(w, h, n, 8, 12)
            L = port.lowres_sample(img)
            lres = port.lowres_encode(L, q)
            unmap = port.mapfun_parse(port.mapfun_serialize(port.lowres_map_table(q)))
            rows, cols = (h + 7) >> 3, (w + 7) >> 3
            want = port.lowres_decode(lres, n, rows, cols, unmap)
            buf = np.zeros((1, (lres.size + 63) & ~63), np.uint8)
            buf[0, : lres.size] = lres
            got = ctx.stage_lres_decode(dev(buf), w, h, n, unmap).cpu().numpy()[0]
            assert_same(got, want, f"lres decode {(w, h, n)} q{q}")
    # arbitrary predictor bytes / deltas (3..253 fall to the default predictor)
    rng = np.random.default_rng(2)
    w, h, n = 136, 264, 2
    rows, cols = 33, 17
    size = port.lowres_channel_size(rows, cols) * n
    lres = rng.integers(0, 256, size, dtype=np.uint8)
    unmap = port.mapfun_parse(port.mapfun_serialize(port.lowres_map_table(30)))
    want = port.lowres_decode(lres, n, rows, cols, unmap)
    buf = np.zeros((1, (size + 63) & ~63), np.uint8)
    buf[0, :size] = lres
    assert_same(ctx.stage_lres_decode(dev(buf), w, h, n, unmap).cpu().numpy()[0], want, "random lres bytes")


@pytest.mark.parametrize("shape", SHAPES)
def test_stage_inverse_random_planes(ctx, port, shape):
    """Random code bytes: exercises the int16 narrowing, clamps and crops."""
    w, h, n = shape
    rng = np.random.default_rng(w * 7 + h)
    rows, cols = (h + 7) >> 3, (w + 7) >> 3
    planes = rng.integers(0, 256, rows * cols * 64 * n, dtype=np.uint8)
    planes[rng.random(planes.size) < 0.6] = 0
    R = rng.integers(0, 256, (n, rows, cols), dtype=np.uint8)
    unmap = port.mapfun_parse(port.mapfun_serialize(port.fullres_map_table()))
    for q, yc in ((50, True), (100, False), (0, True)):
        yc = yc and n >= 3
        sl, sc = port.shift_table(q, 0), port.shift_table(q, 1)
        want = port.fullres_restore(planes, w, h, n, yc, R, sl, sc, unmap)
        got = ctx.stage_inverse(dev(planes[None]), dev(R[None]), w, h, n, yc, sl, sc, unmap).cpu().numpy()[0]
        assert_same(got, want, f"inverse {shape} q{q} ycbcr={yc}")


@pytest.mark.parametrize("shape", [(128, 16, 3), (256, 24, 1), (640, 48, 3), (2176, 16, 3), (1920, 24, 3), (1024, 40, 1),
                                   (4224, 8, 3), (1920, 64, 3), (384, 200, 1), (128, 2056, 3), (3840, 24, 3)])
@pytest.mark.parametrize("kind", ["small", "mixed", "wild"])
def test_stage_inverse_lane_pair_path(ctx, port, shape, kind):
    """Shapes that take the two-blocks-per-thread kernel (cols % 16 == 0): one, two and ragged tile
    rows, several column tiles.  'small' keeps every coefficient inside [-4096, 4095] (packed 16-bit
    arithmetic), 'wild' is random code bytes (every warp falls back to the int32 arithmetic),
    'mixed' has a few large codes so both paths run side by side in one launch."""
    w, h, n = shape
    rng = np.random.default_rng(w + 31 * h + len(kind))
    rows, cols = h >> 3, w >> 3
    size = rows * cols * 64 * n
    if kind == "wild":
        planes = rng.integers(0, 256, size, dtype=np.uint8)
        planes[rng.random(size) < 0.5] = 0
    else:
        planes = rng.choice(np.array([0, 0, 0, 0, 1, 255, 2, 254, 3, 253, 9, 247, 30, 226], np.uint8), size)
        if kind == "mixed":
            idx = rng.integers(0, size, max(1, size // 3000))
            planes[idx] = rng.integers(100, 157, idx.size, dtype=np.uint8)
    R = rng.integers(0, 256, (n, rows, cols), dtype=np.uint8)
    unmap = port.mapfun_parse(port.mapfun_serialize(port.fullres_map_table()))
    for q, yc in ((50, True), (100, False), (0, True)):
        yc = yc and n >= 3
        sl, sc = port.shift_table(q, 0), port.shift_table(q, 1)
        want = port.fullres_restore(planes, w, h, n, yc, R, sl, sc, unmap)
        got = ctx.stage_inverse(dev(planes[None]), dev(R[None]), w, h, n, yc, sl, sc, unmap).cpu().numpy()[0]
        assert_same(got, want, f"inverse {shape} {kind} q{q} ycbcr={yc}")


def test_stage_inverse_many_distinct_shifts(ctx, port):
    """The lane-pair kernel keeps one dequantisation table per DISTINCT shift, at most eight: a stream whose
    (in-band) shift tables use more of them is decoded in the kernel's overflow mode (plain unmap table,
    int32 arithmetic).  Also eight exactly, and small shifts (no pre-division of the tables)."""
    rng = np.random.default_rng(77)
    unmap = port.mapfun_parse(port.mapfun_serialize(port.fullres_map_table()))
    for (w, h, n) in [(640, 48, 3), (1024, 40, 1)]:
        rows, cols = h >> 3, w >> 3
        size = rows * cols * 64 * n
        planes = rng.choice(np.array([0, 0, 0, 0, 1, 255, 2, 254, 3, 253, 9, 247, 30, 226], np.uint8), size)
        R = rng.integers(0, 256, (n, rows, cols), dtype=np.uint8)
        for nshift, base in ((12, 0), (8, 3), (16, 0), (9, 3)):
            sl = ((np.arange(64) * 5) % nshift + base).astype(np.uint8)
            sc = ((np.arange(64) * 7 + 3) % nshift + base).astype(np.uint8)
            sl, sc = np.minimum(sl, 15), np.minimum(sc, 15)
            want = port.fullres_restore(planes, w, h, n, n >= 3, R, sl, sc, unmap)
            got = ctx.stage_inverse(dev(planes[None]), dev(R[None]), w, h, n, n >= 3, sl, sc, unmap).cpu().numpy()[0]
            assert_same(got, want, f"inverse {(w, h, n)} with {nshift} distinct shifts from {base}")


# ---------------------------------------------------------------------------------------------
# whole decoder
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("quality,ycbcr", [(50, True), (5, True), (100, True), (60, False)])
def test_decode_matches_oracle(ctx, port, shape, quality, ycbcr):
    w, h, n = shape
    img = port.synth(w, h, n, 4, 6)
    packed = port.encode(img, quality, ycbcr)
    for flags in (0, 1):
        want = port.decode(packed, strict=(flags == 0))
        got = ctx.decode(packed, flags)
        assert (got is None) == (want is None), f"{shape} q{quality} flags {flags}: reject mismatch"
        if want is not None:
            assert_same(got, want, f"decode {shape} q{quality} flags {flags}")


def test_decode_fixture_bitstreams(ctx, fixtures):
    i = 0
    while f"case{i}_meta" in fixtures:
        if f"case{i}_pixels" in fixtures:
            got = ctx.decode(fixtures[f"case{i}_himg"].tobytes())
            assert got is not None
            assert_same(got, fixtures[f"case{i}_pixels"], f"fixture {i}")
        i += 1


def test_decode_rejects_garbage(ctx, port):
    img = port.synth(64, 48, 3, 1, 6)
    good = port.encode(img, 90, True)
    assert ctx.decode(good) is not None
    assert ctx.decode(b"") is None
    assert ctx.decode(b"RIFF" + b"\0" * 20) is None
    assert ctx.decode(good[:-1]) is None  # RIFF size mismatch
    bad = bytearray(good)
    bad[20] = 2  # version
    assert ctx.decode(bytes(bad)) is None
    rng = np.random.default_rng(0)
    for _ in range(20):  # corrupted payloads must never crash; result may be reject or garbage pixels
        bad = bytearray(good)
        for pos in rng.integers(31, len(good), 8):
            bad[int(pos)] = int(rng.integers(0, 256))
        ctx.decode(bytes(bad))
        ctx.decode(bytes(bad), flags=1)


# ---------------------------------------------------------------------------------------------
# batch API (device resident) + round-trip properties at size
# ---------------------------------------------------------------------------------------------
def test_batch_encode_decode(ctx, port):
    w, h, n = 256, 136, 3
    imgs = np.stack([port.synth(w, h, n, 100 + k, 6) for k in range(9)])
    out, sizes = ctx.encode_batch(dev(imgs), 50, True)
    out_h, sizes_h = out.cpu().numpy(), sizes.cpu().numpy()
    packed = []
    for k in range(9):
        want = port.encode(imgs[k], 50, True)
        assert sizes_h[k] == len(want)
        assert_same(out_h[k, : sizes_h[k]], np.frombuffer(want, np.uint8), f"batch image {k}")
        packed.append(want)
    offsets = torch.arange(9, dtype=torch.int64, device="cuda") * out.stride(0)
    px, status = ctx.decode_batch(out.reshape(-1), offsets, sizes, w, h, n)
    assert int(status.abs().sum().cpu()) == 0
    px = px.cpu().numpy()
    for k in range(9):
        assert_same(px[k], port.decode(packed[k]), f"batch decode {k}")


def test_batch_decode_mixed_quality_and_rejects(ctx, port):
    w, h, n = 128, 64, 3
    streams = [port.encode(port.synth(w, h, n, k, 6), q, yc) for k, (q, yc) in enumerate([(50, True), (95, False), (2, True), (75, True)])]
    streams.append(b"RIFF" + b"\1" * 40)
    streams.append(port.encode(port.synth(64, 64, n, 9, 6), 50, True))  # wrong shape
    offs = np.cumsum([0] + [(len(s) + 15) & ~15 for s in streams])
    buf = np.zeros(offs[-1] + 64, np.uint8)
    for o, s in zip(offs, streams):
        buf[o : o + len(s)] = np.frombuffer(s, np.uint8)
    px, status = ctx.decode_batch(dev(buf), dev(offs[:-1].astype(np.int64)), dev(np.array([len(s) for s in streams], np.int32)), w, h, n)
    status, px = status.cpu().numpy(), px.cpu().numpy()
    for k, s in enumerate(streams[:4]):
        want = port.decode(s)
        assert (status[k] == 0) == (want is not None), f"stream {k}"
        if want is not None:
            assert_same(px[k], want, f"stream {k}")
    assert status[4] != 0 and status[5] != 0


def test_large_batch_round_trip_properties(ctx, port):
    """Full-size c4 slice: a batch of 1080p images; checksum of per-image checksums against the
    oracle for a sample, size-independent properties (determinism, decode(encode) within the
    codec's loss bound, identical results regardless of batch position) for all."""
    w, h, n, B = 1920, 1080, 3, 12
    base = port.synth(w, h, n, 1, 6)
    imgs = np.stack([base if k % 4 == 0 else port.synth(w, h, n, 1 + k, 6) for k in range(B)])
    d = dev(imgs)
    out, sizes = ctx.encode_batch(d, 50, True)
    out2, sizes2 = ctx.encode_batch(d, 50, True)
    assert torch.equal(sizes, sizes2) and torch.equal(out[:, :1024], out2[:, :1024])
    sizes_h = sizes.cpu().numpy()
    out_h = out.cpu().numpy()
    for k in range(0, B, 4):  # same image => same bitstream wherever it sits in the batch
        assert sizes_h[k] == 849760
        assert f"{port.fnv(out_h[k, : sizes_h[k]]):016x}" == "26e587882464e706"
    want1 = port.encode(imgs[1], 50, True)
    assert_same(out_h[1, : sizes_h[1]], np.frombuffer(want1, np.uint8), "image 1")
    offsets = torch.arange(B, dtype=torch.int64, device="cuda") * out.stride(0)
    px, status = ctx.decode_batch(out.reshape(-1), offsets, sizes, w, h, n)
    assert int(status.abs().sum().cpu()) == 0
    px_h = px.cpu().numpy()
    assert f"{port.fnv(px_h[0]):016x}" == "752610ecc81df78e"
    assert_same(px_h[1], port.decode(want1), "decode image 1")
    err = (px_h.astype(np.int32) - imgs.astype(np.int32))
    psnr = 10 * np.log10(255.0 ** 2 / np.mean(err.astype(np.float64) ** 2))
    assert psnr > 30.0, psnr


def test_python_mirror_api(ctx, port):
    import himg_b200

    img = port.synth(64, 48, 3, 1, 6)
    enc = himg_b200.Encoder(ctx)
    assert enc.Encode(img, 64, 48, 3, 3, 95, True)
    assert enc.packed_size() == len(enc.packed_data()) and enc.packed_data() == port.encode(img, 95, True)
    assert port.decode(enc.packed_data()) is not None  # a stream the reference decoder accepts
    dec = himg_b200.Decoder(0, ctx)
    assert dec.Decode(enc.packed_data(), enc.packed_size())
    assert (dec.width(), dec.height(), dec.num_channels()) == (64, 48, 3)
    assert_same(dec.unpacked_data(), port.decode(enc.packed_data()), "mirror decode")
    assert not dec.Decode(b"nope", 4)


def test_host_batch_api_pipelined(ctx, port):
    """himgcu_encode_batch_host / himgcu_decode_batch_host: pinned and pageable host buffers, more
    sub-batches than coding lanes (forced by the smallest staging budget), ragged last sub-batch,
    1 / 2 / 4 lanes."""
    w, h, n, B = 256, 136, 3, 23
    imgs = np.stack([port.synth(w, h, n, 300 + k, 6) for k in range(B)])
    want = [port.encode(imgs[k], 80, True) for k in range(B)]
    ctx.set_option("host_sub_batch_bytes", 1 << 20)  # 4-5 images per sub-batch
    try:
        for lanes, pinned in ((1, False), (2, True), (4, True), (4, False)):
            ctx.set_option("host_lanes", lanes)
            src = torch.from_numpy(imgs).pin_memory() if pinned else imgs
            out, offsets, sizes = ctx.encode_batch_host(src, 80, True)
            out = np.asarray(out)
            for k in range(B):
                assert sizes[k] == len(want[k])
                assert_same(out[int(offsets[k]): int(offsets[k]) + int(sizes[k])], np.frombuffer(want[k], np.uint8), f"host batch image {k}")
            px, status = ctx.decode_batch_host(out, offsets, sizes, w, h, n)
            assert int(np.abs(status).sum()) == 0
            for k in range(B):
                assert_same(px[k], port.decode(want[k]), f"host batch decode {k} ({lanes} lanes)")
    finally:
        ctx.set_option("host_sub_batch_bytes", 64 << 20)
        ctx.set_option("host_lanes", 3)


def test_item_lists_are_an_optimisation_only(port):
    # the packer reads the item lists of the histogram pass (pieces of <= 2048 items) or rebuilds them from
    # the planes (denser pieces, or option item_lists = 0): same bytes either way, sparse to dense content
    import himg_b200

    c = himg_b200.Context(0)
    try:
        imgs = np.stack([port.synth(512, 304, 3, 40 + k, 6 + 30 * k) for k in range(3)])
        for q in (10, 50, 100):
            out = {}
            for flag in (1, 0):
                c.set_option("item_lists", flag)
                o, s = c.encode_batch(dev(imgs), q, True)
                out[flag] = (o.cpu().numpy(), s.cpu().numpy())
            assert np.array_equal(out[0][1], out[1][1])
            for k in range(3):
                n = int(out[1][1][k])
                want = port.encode(imgs[k], q, True)
                assert n == len(want)
                assert_same(out[1][0][k, :n], np.frombuffer(want, np.uint8), f"lists on, q{q} image {k}")
                assert_same(out[0][0][k, :n], out[1][0][k, :n], f"lists off, q{q} image {k}")
    finally:
        c.close()


def test_decode_broken_segment_chain(ctx, port):
    # the segment-header walk of a single image runs inside the decode kernel and publishes entries as it
    # goes: a chain that breaks half way must reject the image (and release every waiting row), never hang
    img = port.synth(256, 400, 3, 3, 6)
    good = port.encode(img, 50, True)
    assert ctx.decode(good) is not None
    at = good.index(b"FRES") + 8
    mid = at + (len(good) - at) // 2
    bad = bytearray(good)
    bad[mid : mid + 8192] = b"\xff" * min(8192, len(good) - mid)
    for flags in (0, 1):
        assert ctx.decode(bytes(bad), flags=flags) is None
    assert port.decode(bytes(bad)) is None
    out = ctx.decode(good)
    assert_same(out, port.decode(good), "decode after a rejected stream")


@pytest.mark.parametrize("nch", [5, 6, 8])
def test_more_than_four_channels(ctx, port, nch):
    # the reference passes any number of channels through (ycbcr.cpp:24-52, encoder.cpp:69): the first three
    # are colour mapped when asked, the others coded as they are
    for (w, h) in [(64, 40), (100, 37)]:
        img = port.synth(w, h, nch, 3, 6)
        for q, yc in [(50, True), (90, False)]:
            want = port.encode(img, q, yc)
            got = ctx.encode(img, q, yc)
            assert_same(np.frombuffer(got, np.uint8), np.frombuffer(want, np.uint8), f"encode {w}x{h}x{nch} q{q} ycbcr={yc}")
            px = ctx.decode(want)
            ref_px = port.decode(want)
            assert (px is None) == (ref_px is None)
            if ref_px is None:
                px, ref_px = ctx.decode(want, flags=1), port.decode(want, strict=False)
            assert_same(px, ref_px, f"decode {w}x{h}x{nch} q{q} ycbcr={yc}")
    imgs = np.stack([port.synth(48, 24, nch, 20 + k, 9) for k in range(3)])
    out, sizes = ctx.encode_batch(dev(imgs), 60, True)
    for k in range(3):
        want = port.encode(imgs[k], 60, True)
        assert int(sizes[k]) == len(want)
        assert_same(out[k, : len(want)].cpu().numpy(), np.frombuffer(want, np.uint8), f"batch image {k}")


def test_generic_kernels_still_match(port):
    """force_generic routes aligned shapes through the generic kernels (k_forward, k_inverse,
    k_huff_hist, k_huff_pack) that normally only see odd shapes; both paths must agree with the
    oracle."""
    import himg_b200

    c = himg_b200.Context(0)
    try:
        c.set_option("force_generic", 1)
        for (w, h, n, q) in [(256, 136, 3, 50), (512, 64, 1, 90), (128, 128, 4, 20)]:
            img = port.synth(w, h, n, 9, 6)
            packed = c.encode(img, q, True)
            assert_same(np.frombuffer(packed, np.uint8), np.frombuffer(port.encode(img, q, True), np.uint8), f"generic encode {(w, h, n, q)}")
            got = c.decode(packed, 1)
            assert_same(got, port.decode(packed, strict=False), f"generic decode {(w, h, n, q)}")
    finally:
        c.close()
