"""Warp-team entropy coder (k_huff_hist4 / k_huff_pack4): framed chunks whose segments are not split
into parts.  Every case is coded with option huff_warp_teams = 2 (warp teams at any batch size) and 0
(k_huff_hist2 / k_huff_pack3); both must give the same bytes, and the oracle's."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def ctxs():
    import himg_b200

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    cs = {}
    for teams in (0, 2):
        c = himg_b200.Context(0)
        c.set_option("huff_warp_teams", teams)
        cs[teams] = c
    yield cs
    for c in cs.values():
        c.close()


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def check_bytes(got, want, what):
    got = np.asarray(got, np.uint8).reshape(-1)
    want = np.asarray(want, np.uint8).reshape(-1)
    assert got.size == want.size, f"{what}: size {got.size} vs {want.size}"
    idx = np.flatnonzero(got != want)
    assert idx.size == 0, f"{what}: {idx.size} bytes differ, first at {idx[0]}"


def huff_both(ctxs, port, data, bs, what):
    """data [n][size] coded in segments of bs bytes with both coders, against the oracle."""
    data = np.ascontiguousarray(data, np.uint8)
    res = {}
    for teams, c in ctxs.items():
        out, sizes = c.stage_huff_compress(dev(data), bs)
        res[teams] = (out.cpu().numpy(), sizes.cpu().numpy())
    for i in range(data.shape[0]):
        want = np.frombuffer(port.huff_compress(data[i], bs), np.uint8)
        for teams in (2, 0):
            out, sizes = res[teams]
            check_bytes(out[i, : sizes[i]], want, f"{what}, item {i}, huff_warp_teams={teams}")


def encode_both(ctxs, port, imgs, q, what):
    res = {}
    for teams, c in ctxs.items():
        out, sizes = c.encode_batch(dev(imgs), q, True)
        res[teams] = (out.cpu().numpy(), sizes.cpu().numpy())
    for k in range(imgs.shape[0]):
        want = np.frombuffer(port.encode(imgs[k], q, True), np.uint8)
        for teams in (2, 0):
            out, sizes = res[teams]
            check_bytes(out[k, : sizes[k]], want, f"{what}, image {k}, huff_warp_teams={teams}")
    return res[2]


@pytest.mark.parametrize("q", [0, 50, 100])
def test_1080p_batch(ctxs, port, q):
    # three 1080p images: 405 segments of 46 080 bytes, enough that the segments get no parts
    imgs = np.stack([port.synth(1920, 1080, 3, 1 + k, 6) for k in range(3)])
    encode_both(ctxs, port, imgs, q, f"1080p q{q}")


def test_random_content(ctxs, port):
    rng = np.random.default_rng(31)
    imgs = rng.integers(0, 256, (3, 480, 640, 3), dtype=np.uint8)
    for q in (20, 50, 100):
        encode_both(ctxs, port, imgs, q, f"random q{q}")


@pytest.mark.parametrize("nch", [1, 2, 3, 4])
def test_channels(ctxs, port, nch):
    # 1016 rows: 127 segments, so that the last CTA of eight segments is partial
    imgs = np.stack([port.synth(256, 1016, nch, 50 + k, 6 + 20 * k) for k in range(2)])
    for q in (10, 60, 100):
        encode_both(ctxs, port, imgs, q, f"{nch} channels q{q}")


def test_batch_position_independence(ctxs, port):
    base = port.synth(512, 200, 3, 3, 6)
    imgs = np.stack([base if k % 3 == 0 else port.synth(512, 200, 3, 10 + k, 6) for k in range(7)])
    out, sizes = encode_both(ctxs, port, imgs, 50, "batch")
    for k in (3, 6):
        assert sizes[k] == sizes[0]
        check_bytes(out[k, : sizes[k]], out[0, : sizes[0]], f"image {k} vs image 0")


def test_sparse_dense_and_empty_segments(ctxs, port):
    rng = np.random.default_rng(32)
    nseg, bs = 13, 4096  # nseg % 8 != 0
    data = rng.integers(0, 256, (3, nseg * bs), dtype=np.uint8)
    dens = rng.random((3, nseg)).repeat(bs, 1)
    data[rng.random(data.shape) < dens] = 0
    data[:, 2 * bs : 3 * bs] = 0  # an all-zero segment
    data[:, 5 * bs : 6 * bs] = rng.integers(1, 256, bs)  # every byte an item: over the list capacity
    data[0, : 4 * bs] = 0  # the first segments of an item empty
    huff_both(ctxs, port, data, bs, "sparse / dense / empty")
    data[:, -1] = 9  # an item in the last byte
    huff_both(ctxs, port, data, bs, "last byte")


def test_incompressible_over_list_capacity(ctxs, port):
    # 16 KiB segments hold up to 4096 items in the list: these have 90 % non-zero bytes
    rng = np.random.default_rng(33)
    data = rng.integers(0, 256, (2, 20 * 16384), dtype=np.uint8)
    data[rng.random(data.shape) < 0.1] = 0
    huff_both(ctxs, port, data, 16384, "incompressible")


def test_long_zero_runs(ctxs, port):
    # runs of 16 662 zeros or more (maximal tokens), in front of an item, at the segment end and over a
    # whole segment; a run of 65 536 or more does not fit the u16 list entry (the packer walks the planes)
    bs, nseg, n = 100000, 40, 8  # 320 segments: no parts
    data = np.zeros((n, nseg * bs), np.uint8)
    rng = np.random.default_rng(34)
    for i in range(n):
        for s in range(nseg):
            seg = data[i, s * bs : (s + 1) * bs]
            kind = (i + s) % 5
            if kind == 0:
                seg[[16661, 16662 + 16661, 70000]] = 7  # runs of exactly 16 661 / 16 661, a tail of 29 999
            elif kind == 1:
                seg[[16662, 2 * 16662 + 1, 99999]] = 3  # exactly one maximal run, then two of 16 662
            elif kind == 2:
                seg[rng.integers(0, 500, 50)] = rng.integers(1, 256, 50)  # a tail of ~99 500 zeros
            elif kind == 3:
                seg[99000] = 1  # a run of 99 000 zeros in front of the only item
            # kind 4: all zero
    huff_both(ctxs, port, data, bs, "long runs")


def test_deep_tree(ctxs, port):
    # Fibonacci symbol counts give codes of up to 26 bits; items of more than 32 and more than 64 bits
    rng = np.random.default_rng(11)
    f = [1, 1]
    while len(f) < 27:
        f.append(f[-1] + f[-2])
    dense = np.concatenate([np.full(f[26 - k] - (2 if k == 22 else 0), k + 1, np.uint8) for k in range(23)])
    rng.shuffle(dense)
    z = lambda n, v: np.r_[np.zeros(n, np.uint8), np.uint8(v)]
    deep = np.concatenate([dense[:1000], [np.uint8(25)], dense[1000:70001], z(5000, 24), dense[70001:300000], z(100, 23),
                           dense[300000:300007], z(200, 23), dense[300007:]])
    bs = 8192
    deep = deep[: deep.size - deep.size % bs]
    huff_both(ctxs, port, deep[None], bs, "deep tree")


def test_item_lists_off(port):
    import himg_b200

    c = himg_b200.Context(0)
    try:
        c.set_option("item_lists", 0)
        c.set_option("huff_warp_teams", 2)
        imgs = np.stack([port.synth(512, 304, 3, 40 + k, 6 + 30 * k) for k in range(3)])
        for q in (10, 50, 100):
            out, sizes = c.encode_batch(dev(imgs), q, True)
            out, sizes = out.cpu().numpy(), sizes.cpu().numpy()
            for k in range(3):
                check_bytes(out[k, : sizes[k]], np.frombuffer(port.encode(imgs[k], q, True), np.uint8), f"q{q} image {k}")
    finally:
        c.close()


def test_default_selection(port):
    # default option: warp teams once the batch has a wave of segments (148 SMs x 32 warps), a CTA per
    # segment below that
    import himg_b200

    rng = np.random.default_rng(35)
    c = himg_b200.Context(0)
    try:
        for nseg in (1000, 5000):
            bs = 512
            data = rng.integers(0, 256, (1, nseg * bs), dtype=np.uint8)
            data[rng.random(data.shape) < 0.85] = 0
            out, sizes = c.stage_huff_compress(dev(data), bs)
            n = int(sizes.cpu()[0])
            check_bytes(out.cpu().numpy()[0, :n], np.frombuffer(port.huff_compress(data[0], bs), np.uint8), f"{nseg} segments")
    finally:
        c.close()
