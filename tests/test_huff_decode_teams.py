"""Parallel Huffman stream decoder (k_dec_stream_par) against the oracle, in every launch shape.

The stage call picks one of six shapes from the batch size, the segment count, the segment size and
force_generic (decode_team / use_decode_cluster in api.cu): warp teams, CTA teams of 64 to 1024
threads, and clusters of 8 CTAs of 256 or 512 threads.  A Python mirror of that choice lists calls
that reach every shape, and a profiled call proves that each one does.  A seeded corpus of streams
built to hit the decoder's paths (multi-token LUT, second-level tables, tree walks, single-leaf trees,
the last-bits rule, zero runs at segment ends, non-resynchronising streams, short streams) goes
through several shapes, and hostile variants of them check the accept / reject decision: every item
must give the oracle's status, strict and lenient, and the oracle's bytes where it accepts."""
import ctypes as C
import json
import re
import tempfile

import numpy as np
import pytest

KB = 1 << 10
RUN_SEG = 32 * KB  # segment size of the rare-runs stream
KLUT, KSUB, KSUBCAP = 11, 5, 64  # kLutBits, kSubBits, kSubCap (huff_dec_kernels.cuh)
RUN_BASE = {256: 2, 257: 3, 258: 7, 259: 23, 260: 279}  # shortest run of each zero-run symbol
EXTRA = {257: 2, 258: 4, 259: 8, 260: 14}  # extra bits after a zero-run symbol


# ---------------------------------------------------------------------------------------------
# mirror of the launch choice of himgcu_stage_huff_uncompress (api.cu)
# ---------------------------------------------------------------------------------------------
def decode_team(streams, out_bytes, base):
    team = base
    while team < 1024 and streams * team < 131072 and out_bytes // (team * 2) >= 256:
        team *= 2
    return team


def stage_shape(n, out_size, block_size, force_generic=False):
    """(template arguments of k_dec_stream_par, threads per CTA) of a stage call."""
    seg = out_size if block_size < 1 else block_size
    nseg = out_size // seg
    if nseg == 1 and n <= 16 and seg >= 64 * KB and not force_generic:
        return "false, 8, 0", 512 if seg >= 256 * KB else 256
    team = decode_team(n * nseg, seg, 256 if nseg == 1 else 32)
    return ("true, 1, 0", 256) if team == 32 else ("false, 1, 0", team)


# (name, n, out_size, block_size, force_generic): every shape the stage call has
MATRIX = [
    ("warp_teams_partial_cta", 3, 13 * 4096, 4096, False),
    ("framed_cta64", 2, 3 * 16 * KB, 16 * KB, False),
    ("framed_cta128", 2, 3 * 32 * KB, 32 * KB, False),
    ("framed_cta256", 2, 2 * 64 * KB, 64 * KB, False),
    ("framed_cta512", 2, 2 * 128 * KB, 128 * KB, False),
    ("framed_cta1024", 1, 2 * 256 * KB, 256 * KB, False),
    ("unframed_cta256", 17, 64 * KB, 0, False),
    ("unframed_cta512", 17, 128 * KB, 0, False),
    ("unframed_cta1024", 1, 256 * KB, 0, True),
    ("cluster256", 2, 64 * KB, 0, False),
    ("cluster512", 1, 256 * KB, 0, False),
    ("one_segment_cta256", 1, 8 * KB, 8 * KB, False),
    ("one_segment_cluster256", 2, 64 * KB, 64 * KB, False),
]
MATRIX_SHAPES = {
    "warp_teams_partial_cta": ("true, 1, 0", 256), "framed_cta64": ("false, 1, 0", 64),
    "framed_cta128": ("false, 1, 0", 128), "framed_cta256": ("false, 1, 0", 256),
    "framed_cta512": ("false, 1, 0", 512), "framed_cta1024": ("false, 1, 0", 1024),
    "unframed_cta256": ("false, 1, 0", 256), "unframed_cta512": ("false, 1, 0", 512),
    "unframed_cta1024": ("false, 1, 0", 1024), "cluster256": ("false, 8, 0", 256), "cluster512": ("false, 8, 0", 512),
    "one_segment_cta256": ("false, 1, 0", 256), "one_segment_cluster256": ("false, 8, 0", 256),
}

# batch sizes tried when a stream is put through several shapes, and the output they may take
BATCHES = (1, 2, 17, 40, 150, 300, 520, 1100, 2100, 4100)
BATCH_BYTES = 128 << 20


def shape_configs(out_size, block_size, limit=3):
    """Up to `limit` (n, force_generic) choices that decode the stream in distinct shapes."""
    seen, out = set(), []
    for n in BATCHES:
        for fg in (False, True):
            s = stage_shape(n, out_size, block_size, fg)
            if n * out_size <= BATCH_BYTES and s not in seen and len(out) < limit:
                seen.add(s)
                out.append((n, fg))
    return out


# ---------------------------------------------------------------------------------------------
# corpus
# ---------------------------------------------------------------------------------------------
def natural_planes(port, q, seed=5, amp=9):
    """FRES planes of a 1024x64 RGB image: 8 block rows of 24 576 bytes."""
    img = port.synth(1024, 64, 3, seed, amp)
    cm = port.rgb_to_ycbcr(img)
    return port.fullres_planes(cm, port.lowres_sample(cm), q, True)


def natural_bytes(port, size):
    p = natural_planes(port, 50)
    return np.resize(p, size)


def fibonacci_deep():
    """The deep-tree construction of test_gpu_parity._huff_cases and test_huff_warp_teams.test_deep_tree: Fibonacci
    counts give codes of up to 26 bits, "5000 zeros + literal 24" is one item of more than 64 bits and "100 zeros +
    literal 23" one of more than 32."""
    rng = np.random.default_rng(11)
    f = [1, 1]
    while len(f) < 27:
        f.append(f[-1] + f[-2])
    dense = np.concatenate([np.full(f[26 - k] - (2 if k == 22 else 0), k + 1, np.uint8) for k in range(23)])
    rng.shuffle(dense)
    z = lambda n, v: np.r_[np.zeros(n, np.uint8), np.uint8(v)]
    deep = np.concatenate([dense[:1000], [np.uint8(25)], dense[1000:70001], z(5000, 24), dense[70001:300000], z(100, 23),
                           dense[300000:300007], z(200, 23), dense[300007:]])
    return deep[: deep.size & ~3]


def geometric(rng, nsym, first=1):
    """Literal first + k occurs 2^(nsym - 1 - k) times (+1 for the last): code lengths 1 .. nsym - 1."""
    d = np.concatenate([np.full(1 << (nsym - 1 - k), first + k, np.uint8) for k in range(nsym)] + [np.uint8([first + nsym - 1])])
    rng.shuffle(d)
    return d


def literals_then_zeros(rng, nseg, bs):
    data = np.zeros((nseg, bs), np.uint8)
    for s in range(nseg):
        m = int(rng.integers(20, 120))
        data[s, :m] = rng.integers(1, 5, m)
    return data.reshape(-1)


def build_corpus(port):
    rng = np.random.default_rng(2024)
    c = {}
    q50, q100 = natural_planes(port, 50), natural_planes(port, 100)
    c["natural_q50"] = (q50, 24576)
    c["natural_q100"] = (q100, 24576)
    c["natural_q50_unframed"] = (q50, 0)
    c["natural_q100_unframed"] = (q100, 0)
    deep = fibonacci_deep()
    c["deep_unframed"] = (deep, 0)
    c["deep_framed"] = (deep[: deep.size - deep.size % (64 * KB)], 64 * KB)
    sc = np.concatenate([np.repeat(np.arange(1, 16, dtype=np.uint8), 24000), np.repeat(np.arange(16, 256, dtype=np.uint8), 100)])
    rng.shuffle(sc)
    c["subcap_overflow"] = (sc, 0)
    c["subcap_overflow_framed"] = (sc, 38400)
    c["window_edges"] = (geometric(rng, 19), 0)  # 2^18 bytes, code lengths 1 .. 18
    c["window_edges_framed"] = (c["window_edges"][0], 16 * KB)
    # dense literals with rare runs: the run symbols get the longest codes, then 8 or 14 extra bits; segment 2
    # of the framed stream ends in a run of 16 662 zeros (one maximal token)
    runs = np.concatenate([geometric(rng, 18), geometric(rng, 18)])  # 2 x 2^17 bytes
    for at, length in ((1000, 300), (40000, 100), (120000, 20000), (RUN_SEG * 3 - 16662, 16662), (200000, 279)):
        runs[at: at + length] = 0
    runs[RUN_SEG * 3] = 9
    c["rare_runs"] = (runs, RUN_SEG)
    c["rare_runs_unframed"] = (runs, 0)
    c["single_leaf"] = (np.full(20000, 7, np.uint8), 0)
    c["single_leaf_framed"] = (np.full(20000, 7, np.uint8), 4000)
    c["single_leaf_run"] = (np.zeros(4000, np.uint8), 400)  # a single run symbol
    c["two_leaf"] = (rng.choice(np.uint8([3, 9]), 40000), 0)
    c["two_leaf_framed"] = (c["two_leaf"][0], 4000)
    # eight literals in turn: every code is 3 bits long, so a decoder started 32 k bits into the stream is out
    # of phase for good unless 3 divides k
    per = np.tile(np.arange(1, 9, dtype=np.uint8), 256 * KB // 8)
    c["periodic"] = (per, 0)
    c["periodic_framed"] = (per, 32 * KB)
    c["tiny"] = (np.uint8([1, 2, 3, 1] * 10), 0)  # 80 payload bits: only lane 0 has work
    c["tiny_framed"] = (rng.integers(1, 5, 64).astype(np.uint8), 8)
    eight = rng.integers(1, 9, 5 * 1368).astype(np.uint8)
    c["just_above_warp_subsequences"] = (eight, 1368)  # 4104 bits = 128 x 32 + 8 per segment
    c["just_above_cta256_subsequences"] = (rng.integers(1, 9, 10924).astype(np.uint8), 0)  # 32 772 = 128 x 256 + 4
    # a few literals, then zeros to the end of the segment: in some segments the last multi-token group (a literal
    # and the final zero run) starts in one warp lane's subsequence and its run starts in the next one
    c["last_group_straddles"] = (literals_then_zeros(np.random.default_rng(7), 24, 512), 512)
    return c


_CORPUS = {}


def corpus(port):
    if not _CORPUS:
        _CORPUS.update(build_corpus(port))
    return _CORPUS


def code_lengths(port, data, bs):
    _, code, ln, _ = port.huff_tree(port.huff_histogram(data, bs))
    return code, ln


def payload_bits(port, data, bs):
    """Bits of every segment's payload (before padding)."""
    _, ln = code_lengths(port, data, bs)
    seg = bs if bs > 0 else data.size
    cost = ln.astype(np.int64) + np.array([EXTRA.get(s, 0) for s in range(261)], np.int64)
    return [int((port.huff_histogram(data[k: k + seg], 0).astype(np.int64) * cost).sum()) for k in range(0, data.size, seg)]


def tokens(seg):
    """(symbol, output bytes) of the tokens the encoder cuts a segment into (zero runs greedily)."""
    out, k = [], 0
    while k < seg.size:
        if seg[k]:
            out.append((int(seg[k]), 1))
            k += 1
            continue
        z = 1
        while z < 16662 and k + z < seg.size and seg[k + z] == 0:
            z += 1
        out.append((0 if z == 1 else max(s for s, b in RUN_BASE.items() if b <= z), z))
        k += z
    return out


def straddling_last_groups(port, data, bs, team):
    """Segments whose last multi-token group (as the write pass takes groups: whole tokens inside the kLutBits window,
    at most two non-zero literals, a zero run whose extra bits leave the window ends it) starts in one thread's
    subsequence and has a token that starts in the next.  The thread that takes the group must write all of it."""
    _, _, ln, _ = port.huff_tree(port.huff_histogram(data, bs))
    hits = []
    for si, k in enumerate(range(0, data.size, bs)):
        toks = tokens(data[k: k + bs])
        starts, pos = [], 0
        for sym, _ in toks:
            starts.append(pos)
            pos += int(ln[sym]) + EXTRA.get(sym, 0)
        total = 8 * ((pos + 7) // 8)
        sub = max((-(-total // team) + 31) & ~31, 128)

        def group(i):  # tokens of the group that starts at token i
            p, nlit, j = 0, 0, i
            while j < len(toks) and p < KLUT:
                sym = toks[j][0]
                L, nx = int(ln[sym]), EXTRA.get(sym, 0)
                if L > KLUT - p:
                    break
                if L + nx > KLUT - p:
                    return j - i + 1
                if 0 < sym <= 255:
                    if nlit == 2:
                        break
                    nlit += 1
                p += L + nx
                j += 1
            return j - i

        i = 0
        while i < len(toks):
            g = group(i) if starts[i] + KLUT + 14 <= total else 0
            if g and i + g == len(toks):
                bound = (starts[i] // sub + 1) * sub
                if any(starts[j] >= bound for j in range(i + 1, i + g)):
                    hits.append(si)
            i += max(g, 1)
    return hits


def test_corpus_properties(port):
    """Each corpus stream has the property it is meant to exercise (CPU only)."""
    c = corpus(port)
    for name, (data, bs) in c.items():
        assert data.size % 4 == 0 and (bs == 0 or (bs % 4 == 0 and data.size % bs == 0)), name
        packed = port.huff_compress(data, bs)
        assert np.array_equal(oracle_expect(port, packed, data.size, bs, False), data), name
        # strict mode decodes it too (a framed chunk must be larger than its block size, see segtab_walk), except
        # a single-leaf tree, whose 1-bit codes the reference's decoder does not read
        assert (oracle_expect(port, packed, data.size, bs, True) is None) == name.startswith("single_leaf"), name
    for name in ("natural_q50", "natural_q100"):
        _, ln = code_lengths(port, *c[name])
        assert (ln > 0).sum() > 100, name
    # deep tree: codes longer than the window plus the second-level table, items over 32 and 64 bits
    _, ln = code_lengths(port, c["deep_unframed"][0], 0)
    assert ln.max() == 26 and ln[24] + ln[260] + 14 > 64 and ln[23] + ln[259] + 8 > 32
    # more than kSubCap depth-11 nodes: those beyond it have no second-level table
    code, ln = code_lengths(port, c["subcap_overflow"][0], 0)
    assert sorted(np.bincount(ln)[1:].nonzero()[0] + 1) == [4, 11, 12]
    assert len({int(code[s]) & 0x7FF for s in range(261) if ln[s] == 12}) > KSUBCAP
    # codes of exactly the window, one more, the window plus the second level, one more
    _, ln = code_lengths(port, c["window_edges"][0], 0)
    assert {11, 12, 16, 17} <= set(ln.tolist())
    # rare runs: run symbols with codes over 16 bits and 8 / 14 extra bits, a run ending at a segment end
    data, bs = c["rare_runs"]
    _, ln = code_lengths(port, data, bs)
    assert ln[259] > KLUT + KSUB and ln[260] > KLUT + KSUB
    assert bs == RUN_SEG and not data[3 * bs - 16662: 3 * bs].any() and data[3 * bs - 16663] and data[3 * bs]
    for name, leaves in (("single_leaf", 1), ("single_leaf_framed", 1), ("single_leaf_run", 1), ("two_leaf", 2)):
        _, ln = code_lengths(port, *c[name])
        assert (ln > 0).sum() == leaves, name
    # periodic: one code length, odd, so that subsequence starts (multiples of 32 bits) fall out of phase
    _, ln = code_lengths(port, *c["periodic"])
    assert set(ln[ln > 0].tolist()) == {3}
    assert max(payload_bits(port, *c["tiny"])) < 128 and max(payload_bits(port, *c["tiny_framed"])) < 128
    assert all(128 * 32 < b <= 128 * 32 + 32 for b in payload_bits(port, *c["just_above_warp_subsequences"]))
    assert all(128 * 256 < b <= 128 * 256 + 32 for b in payload_bits(port, *c["just_above_cta256_subsequences"]))
    data, bs = c["last_group_straddles"]
    assert stage_shape(1, data.size, bs) == ("true, 1, 0", 256) and len(straddling_last_groups(port, data, bs, 32)) >= 3
    # the large streams reach more than one shape
    for name, (data, bs) in c.items():
        if data.size >= 64 * KB and (bs == 0 or bs >= 16 * KB):
            assert len(shape_configs(data.size, bs)) >= 2, name


def test_shape_matrix_mirror():
    """The matrix names every shape, and the mirror of the launch choice maps each entry to the one listed."""
    got = {name: stage_shape(n, out, bs, fg) for name, n, out, bs, fg in MATRIX}
    assert got == MATRIX_SHAPES
    assert set(got.values()) == {("true, 1, 0", 256), ("false, 8, 0", 256), ("false, 8, 0", 512)} | {
        ("false, 1, 0", t) for t in (64, 128, 256, 512, 1024)}


def single_leaf_tree(sym):
    """Serialised single-leaf tree (leaf bit, 9-bit symbol, LSB first), padded to bytes."""
    v = 1 | (sym << 1)
    return bytes([v & 255, v >> 8])


def empty_segment_chunks():
    """80 output bytes in 20 segments of 4: chunks whose segments are (mostly) empty."""
    z = b"\0\0" * 20
    return [
        single_leaf_tree(7) + z,  # 0-bit codes: strict mode decodes 4 x literal 7 from nothing
        single_leaf_tree(256) + z,  # a run of two zeros, no extra bits
        single_leaf_tree(257) + z,  # a run with 2 extra bits: they are missing
        single_leaf_tree(300) + z,  # no such symbol
        single_leaf_tree(7) + b"\0\0" * 19,  # a header missing
        single_leaf_tree(7) + b"\x01\x00\x00" + b"\0\0" * 19,  # one segment of 1 byte
        single_leaf_tree(7) + b"\x01\x00\x0f" * 20,  # what the encoder writes: 4 x 1 bit per segment
        (0b10 | 7 << 2 | 1 << 11 | 9 << 12).to_bytes(3, "little") + z,  # two leaves (literals 7, 9): 1-bit codes
    ]


def test_empty_segment_oracle(port):
    """The oracle's decisions that the decoder must follow on empty segments."""
    assert port.huff_compress(np.full(80, 7, np.uint8), 4)[:2] == single_leaf_tree(7)
    chunks = empty_segment_chunks()
    want = [(True, False), (True, False), (False, False), (False, False), (False, False), (False, False), (False, True),
            (False, False)]
    for k, ch in enumerate(chunks):
        got = tuple(oracle_expect(port, ch, 80, 4, strict) is not None for strict in (True, False))
        assert got == want[k], k
    assert np.array_equal(oracle_expect(port, chunks[0], 80, 4, True), np.full(80, 7, np.uint8))
    assert np.array_equal(oracle_expect(port, chunks[1], 80, 4, True), np.zeros(80, np.uint8))


# ---------------------------------------------------------------------------------------------
# helpers: oracle and stage call
# ---------------------------------------------------------------------------------------------
def oracle_expect(port, packed, out_size, bs, strict):
    """What the oracle decodes from one item: the bytes, or None where a segment is rejected."""
    packed = bytes(packed)
    if bs < 1:
        return port.huff_uncompress(packed, out_size, 0, -1, strict=strict, unpacked_total=out_size)
    parts = []
    for b in range(out_size // bs):
        r = port.huff_uncompress(packed, bs, bs, b, strict=strict, unpacked_total=out_size)
        if r is None:
            return None
        parts.append(r)
    return np.concatenate(parts)


def pack_items(items, odd_stride=True):
    """Items (bytes) into one [n][stride] buffer, stride odd when asked."""
    stride = max(len(p) for p in items) + 8
    stride += (stride % 2 == 0) if odd_stride else 0
    buf = np.zeros((len(items), stride), np.uint8)
    for i, p in enumerate(items):
        buf[i, : len(p)] = np.frombuffer(p, np.uint8)
    return buf, np.array([len(p) for p in items], np.int32)


def check_items(got, status, want, what):
    for i, w in enumerate(want):
        assert (int(status[i]) == 0) == (w is not None), f"{what}, item {i}: status {int(status[i])}, oracle {'accepts' if w is not None else 'rejects'}"
        if w is not None:
            d = np.flatnonzero(got[i] != w)
            assert d.size == 0, f"{what}, item {i}: {d.size} bytes differ, first at {d[0]}"


# ---------------------------------------------------------------------------------------------
# GPU tests
# ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ctxs():
    torch = pytest.importorskip("torch")
    import himg_b200

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    cs = {}
    for fg in (False, True):
        c = himg_b200.Context(0)
        c.set_option("force_generic", int(fg))
        cs[fg] = c
    yield cs
    for c in cs.values():
        c.close()


def dev(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def stage(ctx, buf, sizes, out_size, bs, strict):
    out, status = ctx.stage_huff_uncompress(dev(buf), dev(sizes), out_size, bs, 0 if strict else 1)
    return out.cpu().numpy(), status.cpu().numpy()


def decode_same(ctxs, port, packed, out_size, bs, n, fg, what, want=None):
    """n copies of one stream, strict and lenient, against the oracle."""
    buf, sizes = pack_items([packed] * n)
    for strict in (True, False):
        w = want[strict] if want else oracle_expect(port, packed, out_size, bs, strict)
        got, status = stage(ctxs[fg], buf, sizes, out_size, bs, strict)
        check_items(got, status, [w] * n, f"{what} n={n} force_generic={fg} strict={strict}")


def traced_shapes(fn):
    """(template arguments, block size) of every k_dec_stream_par launch of fn(), from a torch.profiler trace."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    with tempfile.NamedTemporaryFile(suffix=".json") as tmp:
        prof.export_chrome_trace(tmp.name)
        events = json.load(open(tmp.name))["traceEvents"]
    out = []
    for e in events:
        if e.get("cat") == "kernel" and "k_dec_stream_par" in e.get("name", ""):
            m = re.search(r"k_dec_stream_par<([^>]*)>", e["name"])
            out.append((m.group(1) if m else e["name"], tuple(e.get("args", {}).get("block", ()))))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("entry", MATRIX, ids=[m[0] for m in MATRIX])
def test_shape_matrix(ctxs, port, entry):
    """Each matrix entry launches the shape the mirror names, and decodes as the oracle does."""
    name, n, out_size, bs, fg = entry
    data = natural_bytes(port, out_size)
    packed = port.huff_compress(data, bs)
    buf, sizes = pack_items([packed] * n)
    launches = traced_shapes(lambda: stage(ctxs[fg], buf, sizes, out_size, bs, False))
    tmpl, team = MATRIX_SHAPES[name]
    assert launches == [(tmpl, (team, 1, 1))], f"{name}: k_dec_stream_par launches {launches}"
    decode_same(ctxs, port, packed, out_size, bs, n, fg, name)
    if bs == out_size:  # one segment, framed: what the oracle decides for a stream whose packed size exceeds it
        noise = np.random.default_rng(n).integers(0, 256, out_size).astype(np.uint8)
        decode_same(ctxs, port, port.huff_compress(noise, 0), out_size, bs, n, fg, name + " incompressible")


CORPUS_NAMES = [
    "natural_q50", "natural_q100", "natural_q50_unframed", "natural_q100_unframed", "deep_unframed", "deep_framed",
    "subcap_overflow", "subcap_overflow_framed", "window_edges", "window_edges_framed", "rare_runs", "rare_runs_unframed",
    "single_leaf", "single_leaf_framed", "single_leaf_run", "two_leaf", "two_leaf_framed", "periodic", "periodic_framed",
    "tiny", "tiny_framed", "just_above_warp_subsequences", "just_above_cta256_subsequences", "last_group_straddles",
]


def test_corpus_names(port):
    assert sorted(CORPUS_NAMES) == sorted(corpus(port))


@pytest.mark.gpu
@pytest.mark.parametrize("name", CORPUS_NAMES)
def test_corpus_across_shapes(ctxs, port, name):
    """The same stream, copied to n items, decodes to the oracle's bytes and status in every shape it reaches."""
    data, bs = corpus(port)[name]
    packed = port.huff_compress(data, bs)
    want = {strict: oracle_expect(port, packed, data.size, bs, strict) for strict in (True, False)}
    for n, fg in shape_configs(data.size, bs):
        decode_same(ctxs, port, packed, data.size, bs, n, fg, name, want)


def segment_headers(packed, data_off, nseg):
    """(position, header bytes, payload size) of each segment of a framed chunk."""
    out, pos = [], data_off
    for _ in range(nseg):
        sz = packed[pos] | packed[pos + 1] << 8
        hl = 2
        if sz & 0x8000:
            sz = (sz & 0x7FFF) | (packed[pos + 2] | packed[pos + 3] << 8) << 15
            hl = 4
        out.append((pos, hl, sz))
        pos += hl + sz
    return out


def header(size, four):
    if not four:
        return bytes([size & 255, size >> 8])
    lo = (size & 0x7FFF) | 0x8000
    return bytes([lo & 255, lo >> 8, (size >> 15) & 255, size >> 23])


def padding_set(port, packed, out_size, bs):
    """The chunk with every padding bit of its last byte set (the bits the oracle's decode does not read)."""
    p = bytearray(packed)
    want = oracle_expect(port, bytes(p), out_size, bs, True)
    for bit in range(7, -1, -1):
        q = bytearray(p)
        q[-1] |= 1 << bit
        if q == p:
            continue
        r = oracle_expect(port, bytes(q), out_size, bs, True)
        if r is None or not np.array_equal(r, want):
            break
        p = q
    return bytes(p)


def hostile_items(port, data, bs, seed):
    """Variants of the stream of (data, bs), each decoded as out_size = data.size with block size bs."""
    rng = np.random.default_rng(seed)
    packed = port.huff_compress(data, bs)
    tree_bytes = (port.huff_tree(port.huff_histogram(data, bs))[0] + 7) // 8
    seg = bs if bs > 0 else data.size
    rows = data.reshape(-1, seg)
    items = {"original": packed, "truncated": packed[:-1], "appended": packed + b"\xa5"}
    items["padding_set"] = padding_set(port, packed, data.size, bs)
    flips = np.frombuffer(packed, np.uint8).copy()
    pos = rng.choice(np.arange(8 * tree_bytes, 8 * len(packed)), min(50, 8 * (len(packed) - tree_bytes) // 4), replace=False)
    np.bitwise_xor.at(flips, pos >> 3, (1 << (pos & 7)).astype(np.uint8))
    items["bit_flips"] = flips.tobytes()
    items["4_bytes_short"] = port.huff_compress(rows[:, :-4].reshape(-1), bs - 4 if bs else 0)
    longer = np.concatenate([rows, np.tile(np.uint8([5, 0, 0, 6]), (rows.shape[0], 1))], 1).reshape(-1)
    items["4_bytes_long"] = port.huff_compress(longer, bs + 4 if bs else 0)
    if bs:
        hdr = segment_headers(packed, tree_bytes, data.size // bs)
        k = len(hdr) // 2
        p, hl, sz = hdr[k]
        for d, tag in ((1, "header_plus_1"), (-1, "header_minus_1")):
            items[tag] = packed[:p] + header(sz + d, hl == 4) + packed[p + hl:]
        items["empty_segment"] = packed[:p] + b"\0\0" + packed[p + hl + sz:]
        p0, hl0, sz0 = hdr[0]
        items["first_segment_empty"] = packed[:p0] + b"\0\0" + packed[p0 + hl0 + sz0:]
    items["original_again"] = packed
    return list(items.items())


HOSTILE = ["natural_q50", "natural_q50_unframed", "deep_unframed", "deep_framed", "subcap_overflow_framed", "rare_runs",
           "window_edges", "periodic_framed", "two_leaf_framed", "single_leaf_framed", "tiny_framed",
           "just_above_warp_subsequences"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", HOSTILE)
def test_hostile_variants(ctxs, port, name):
    """A batch with a different variant in every item: each item gets the oracle's status (and bytes where it
    accepts), whatever its neighbours are, in every shape the batch reaches."""
    data, bs = corpus(port)[name]
    items = hostile_items(port, data, bs, seed=len(name))
    buf, sizes = pack_items([p for _, p in items])
    for strict in (True, False):
        want = [oracle_expect(port, p, data.size, bs, strict) for _, p in items]
        assert want[-1] is not None or (strict and name.startswith("single_leaf"))
        for fg in (False, True):
            got, status = stage(ctxs[fg], buf, sizes, data.size, bs, strict)
            for i, (tag, _) in enumerate(items):
                check_items(got[i: i + 1], status[i: i + 1], want[i: i + 1], f"{name} {tag} force_generic={fg} strict={strict}")


@pytest.mark.gpu
def test_empty_segments(ctxs, port):
    """Empty segments decode where the oracle decodes them: a single-leaf tree in strict mode spends 0 bits per
    token, so 20 empty segments give 20 x 4 copies of its literal."""
    chunks = empty_segment_chunks()
    buf, sizes = pack_items(chunks)
    for strict in (True, False):
        want = [oracle_expect(port, ch, 80, 4, strict) for ch in chunks]
        got, status = stage(ctxs[False], buf, sizes, 80, 4, strict)
        check_items(got, status, want, f"empty segments strict={strict}")


@pytest.mark.gpu
def test_batch_of_distinct_streams(ctxs, port):
    """A different stream in every item (distinct packed sizes, odd row stride), framed and unframed."""
    datas = [natural_planes(port, q, seed=s) for q, s in ((10, 1), (50, 2), (75, 3), (100, 4), (30, 5), (90, 6))]
    for bs in (24576, 0):
        packed = [port.huff_compress(d, bs) for d in datas]
        assert len({len(p) for p in packed}) == len(packed)
        buf, sizes = pack_items(packed)
        assert buf.shape[1] % 2 == 1
        out_size = datas[0].size
        for fg in (False, True):
            for strict in (True, False):
                got, status = stage(ctxs[fg], buf, sizes, out_size, bs, strict)
                check_items(got, status, [oracle_expect(port, p, out_size, bs, strict) for p in packed],
                            f"distinct streams bs={bs} force_generic={fg} strict={strict}")
                if not strict:
                    assert not status.any()


# segment sizes = 4, 8 and 12 (mod 16) and output sizes that are not multiples of 32: byte zero-fill, segments
# that do not start on a 16-byte boundary (unbuffered stores)
ALIGN = [(2, 3 * (16 * KB + 4), 16 * KB + 4), (2, 3 * (32 * KB + 8), 32 * KB + 8), (2, 13 * 4108, 4108),
         (2, 2 * (128 * KB + 12), 128 * KB + 12), (2, 64 * KB + 4, 0), (17, 128 * KB + 12, 0), (1, 256 * KB + 8, 0)]


@pytest.mark.gpu
@pytest.mark.parametrize("n,out_size,bs", ALIGN)
def test_unaligned_segments(ctxs, port, n, out_size, bs):
    assert out_size % 32 and (bs == 0 or bs % 16 in (4, 8, 12))
    data = natural_bytes(port, out_size)
    for fg in (False, True):
        decode_same(ctxs, port, port.huff_compress(data, bs), out_size, bs, n, fg, f"unaligned {out_size}/{bs}")


@pytest.mark.gpu
@pytest.mark.parametrize("out_size,bs,fg", [(3 * (16 * KB + 4), 16 * KB + 4, False), (13 * 4108, 4108, False),
                                            (64 * KB + 4, 0, False), (256 * KB + 4, 0, True)])
def test_raw_output_stride(ctxs, port, out_size, bs, fg):
    """The raw ABI with an output base and stride = 4 (mod 16) into a sentinel-filled buffer: the spans are the
    oracle's bytes and every byte outside them keeps its sentinel."""
    import torch

    n, base = 3, 4
    stride = out_size + ((4 - out_size) % 16) + 16
    assert stride % 16 == 4
    rng = np.random.default_rng(out_size)
    datas = [natural_bytes(port, out_size), rng.integers(0, 256, out_size).astype(np.uint8), natural_bytes(port, out_size)[::-1].copy()]
    packed = [port.huff_compress(d, bs) for d in datas]
    buf, sizes = pack_items(packed)
    ctx = ctxs[fg]
    d_in, d_sizes = dev(buf), dev(sizes)
    out = torch.full((base + n * stride + 64,), 0xA5, dtype=torch.uint8, device="cuda")
    status = torch.full((n,), -1, dtype=torch.int32, device="cuda")
    ctx._bind(d_in, d_sizes, out, status)
    ctx._check(ctx.lib.himgcu_stage_huff_uncompress(ctx.h, d_in.data_ptr(), buf.shape[1], d_sizes.data_ptr(), n, out_size, bs, 0,
                                                    C.c_void_p(out.data_ptr() + base), stride, status.data_ptr()))
    torch.cuda.synchronize()
    got, st = out.cpu().numpy(), status.cpu().numpy()
    inside = np.zeros(got.size, bool)
    for i in range(n):
        inside[base + i * stride: base + i * stride + out_size] = True
        w = oracle_expect(port, packed[i], out_size, bs, True)
        assert (st[i] == 0) == (w is not None), f"item {i}: status {st[i]}"
        if w is not None:
            assert np.array_equal(got[base + i * stride: base + i * stride + out_size], w), f"item {i}"
    outside = np.flatnonzero(~inside & (got != 0xA5))
    assert outside.size == 0, f"{outside.size} bytes outside the output spans written, first at {outside[0]}"
