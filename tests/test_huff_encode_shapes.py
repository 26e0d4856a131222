"""Huffman encoder (k_huff_hist* / k_huff_pack* / k_huff_stale) against the oracle, in every launch shape.

huff_encode_items (api.cu) codes a chunk with the first-generation pair (force_generic), a CTA per segment or per
part of a segment (k_huff_hist2 / k_huff_pack3; a segment is split into 1 to 64 parts when the batch alone cannot
fill the GPU), or warp teams (k_huff_hist4 / k_huff_pack4, framed chunks without parts), with or without the item
lists the histogram pass hands to the packer; k_huff_stale then fills the padding bits of every framed segment.  A
Python mirror of that choice lists stage and image calls that reach every shape, and a profiled call proves that
each one does (kernel names, grids and blocks).  A CPU model of the part bit counts (a zero run counts in the part
of the item that ends it, a run still open at the segment end in the last part) is pinned to the oracle, and a
seeded corpus of streams built for one seam each (runs across parts, greedy 16 662-zero cuts, bytes shared by two
parts, zero-bit parts, pieces at the item-list capacity, u16 run limits of the warp teams, odd segment sizes and
input strides, 27..32-bit codes and items over 64 bits, stale padding from beyond the shared-memory window) is
coded in every shape it reaches.  Every call goes through the raw C ABI into a sentinel-filled buffer whose row
stride is 3 (mod 16), every item must be the oracle's bytes with the sentinel intact behind it, and the device error
flag is read after every call."""
import json
import re
import tempfile
from typing import NamedTuple

import numpy as np
import pytest

KB = 1 << 10
MIB = 1 << 20
MAX_RUN = 16662  # kMaxRun: zeros of one maximal run token
PIECE = 8 * KB  # kTokPiece
ITEM_CAP = 2048  # kItemCap: items of a stored piece list
TEAM_WARPS = 8  # kTeamWarps
SMS = 148
WAVE = SMS * TEAM_WARPS * 4  # resident warps of k_huff_pack4 (kP4MinCtas = 4)
STALE_WINDOW = 1024  # kStaleWindow
LOOKBACK = 2 * KB  # window of zeros_before
SENTINEL = 0xA5
EXTRA = np.array([0] * 257 + [2, 4, 8, 14], np.int64)  # extra bits after each symbol
OK, ERR_CAPACITY, ERR_UNSUPPORTED = 0, 4, 5


# ---------------------------------------------------------------------------------------------
# mirror of the launch choice of huff_encode_items (api.cu)
# ---------------------------------------------------------------------------------------------
class Shape(NamedTuple):
    hist: str
    pack: str
    nsub: int
    sub_size: int
    grid: tuple  # of the histogram and pack launches
    block: int
    stale: tuple  # grid of k_huff_stale (block 256), or None
    pieces_per_part: int  # item-list slots per (segment, part); 0 without lists


def chunk_shape(n, seg_size, nseg, generic=False, teams=1, lists=True):
    nsub, sub = 1, seg_size
    ctas, fill = n * nseg, (SMS * 8 if nseg == 1 else SMS * 2)
    if not generic and ctas < fill and seg_size > 2 * PIECE:
        want = min(64, -(-fill // ctas))
        sub = -(-(-(-seg_size // want)) // PIECE) * PIECE
        nsub = -(-seg_size // sub)
    warp = not generic and nseg > 1 and nsub == 1 and (teams == 2 or (teams == 1 and n * nseg >= WAVE))
    stale = (-(-nseg // 256), n, 1) if nseg > 1 else None
    ppp = -(-sub // PIECE) if lists and not generic else 0
    if generic:
        return Shape("k_huff_hist", "k_huff_pack", 1, seg_size, (nseg, n, 1), 512, stale, ppp)
    if warp:
        return Shape("k_huff_hist4", "k_huff_pack4", 1, seg_size, (-(-nseg // TEAM_WARPS), n, 1), 256, stale, ppp)
    return Shape("k_huff_hist2", "k_huff_pack3", nsub, sub, (nseg * nsub, n, 1), 256, stale, ppp)


def stage_shape(n, in_size, bs, generic=False, teams=1, lists=True):
    """The shape of himgcu_stage_huff_compress(n items of in_size bytes, block size bs)."""
    seg = bs if bs > 0 else in_size
    return chunk_shape(n, seg, in_size // seg, generic, teams, lists)


def image_geom(w, h, nch):
    """(lres_size, seg, rows) of make_geom (common.cuh)."""
    rows, cols = (h + 7) >> 3, (w + 7) >> 3
    return (((rows + 15) // 16) * ((cols + 15) // 16) + rows * cols) * nch, cols * 64 * nch, rows


def image_shapes(n, w, h, nch, generic=False, teams=1, lists=True):
    """The shapes of the two chunks of himgcu_encode_batch: the low-res chunk (one unframed segment) and the FRES
    planes (a segment per block row)."""
    lres, seg, rows = image_geom(w, h, nch)
    return chunk_shape(n, lres, 1, generic, teams, lists), chunk_shape(n, seg, rows, generic, teams, lists)


def launches(shapes):
    """(kernel, grid, block) of the histogram, pack and stale launches of a call coding chunks of these shapes."""
    out = [(s.hist, s.grid, (s.block, 1, 1)) for s in shapes]
    for s in shapes:
        out.append((s.pack, s.grid, (s.block, 1, 1)))
        if s.stale:
            out.append(("k_huff_stale", s.stale, (256, 1, 1)))
    return out


OPTIONS = {  # context name -> (force_generic, huff_warp_teams, item_lists)
    "default": (False, 1, True), "teams": (False, 2, True), "ctas": (False, 0, True), "generic": (True, 1, True),
    "nolists": (False, 1, False), "nolists_teams": (False, 2, False),
}


def shape_of(kind, args, opt):
    g, t, l = OPTIONS[opt]
    return stage_shape(*args, g, t, l) if kind == "stage" else image_shapes(*args, g, t, l)


# (name, kind, args, context): stage args (n, in_size, block_size), image args (n, w, h, nch)
MATRIX = [
    ("unframed_64_parts", "stage", (1, MIB, 0), "default"),
    ("unframed_9_parts_short_last", "stage", (1, 70000, 0), "default"),
    ("unframed_2_parts", "stage", (600, 100000, 0), "default"),
    ("unframed_no_parts_16k", "stage", (3, 16 * KB, 0), "default"),
    ("unframed_no_parts_full_batch", "stage", (1184, 20000, 0), "default"),
    ("framed_3_parts", "stage", (1, 5 * 20000, 20000), "default"),
    ("framed_2_parts", "stage", (2, 100 * 24576, 24576), "default"),
    ("framed_cta_no_parts", "stage", (3, 100 * 24576, 24576), "default"),
    ("teams_option1_partial_cta", "stage", (37, 131 * 1000, 1000), "default"),
    ("teams_option2", "stage", (2, 13 * 4096, 4096), "teams"),
    ("first_generation", "stage", (2, 3 * 20000, 20000), "generic"),
    ("first_generation_unframed", "stage", (1, 70000, 0), "generic"),
    ("lists_off_parts", "stage", (1, 70000, 0), "nolists"),
    ("lists_off_teams", "stage", (2, 13 * 4096, 4096), "nolists_teams"),
    ("image_fres_3_parts_n1", "image", (1, 1024, 64, 3), "default"),
    ("image_fres_3_parts_n12", "image", (12, 1024, 64, 3), "default"),
    ("image_fres_2_parts", "image", (20, 1024, 64, 3), "default"),
    ("image_fres_no_parts", "image", (40, 1024, 64, 3), "default"),
    ("image_1080p_lres_12_parts", "image", (1, 1920, 1080, 3), "default"),
    ("image_4096_gray_lres_parts", "image", (1, 4096, 4096, 1), "default"),
    ("image_lres_2_parts_fres_teams", "image", (600, 1024, 1024, 1), "default"),
    ("image_generic", "image", (2, 1024, 64, 3), "generic"),
]

# (histogram kernel, parts, part size, histogram grid, stale grid) of every entry, per chunk for images
MATRIX_SHAPES = {
    "unframed_64_parts": ("k_huff_hist2", 64, 16 * KB, (64, 1, 1), None),
    "unframed_9_parts_short_last": ("k_huff_hist2", 9, 8 * KB, (9, 1, 1), None),
    "unframed_2_parts": ("k_huff_hist2", 2, 56 * KB, (2, 600, 1), None),
    "unframed_no_parts_16k": ("k_huff_hist2", 1, 16 * KB, (1, 3, 1), None),
    "unframed_no_parts_full_batch": ("k_huff_hist2", 1, 20000, (1, 1184, 1), None),
    "framed_3_parts": ("k_huff_hist2", 3, 8 * KB, (15, 1, 1), (1, 1, 1)),
    "framed_2_parts": ("k_huff_hist2", 2, 16 * KB, (200, 2, 1), (1, 2, 1)),
    "framed_cta_no_parts": ("k_huff_hist2", 1, 24576, (100, 3, 1), (1, 3, 1)),
    "teams_option1_partial_cta": ("k_huff_hist4", 1, 1000, (17, 37, 1), (1, 37, 1)),
    "teams_option2": ("k_huff_hist4", 1, 4096, (2, 2, 1), (1, 2, 1)),
    "first_generation": ("k_huff_hist", 1, 20000, (3, 2, 1), (1, 2, 1)),
    "first_generation_unframed": ("k_huff_hist", 1, 70000, (1, 1, 1), None),
    "lists_off_parts": ("k_huff_hist2", 9, 8 * KB, (9, 1, 1), None),
    "lists_off_teams": ("k_huff_hist4", 1, 4096, (2, 2, 1), (1, 2, 1)),
    "image_fres_3_parts_n1": (("k_huff_hist2", 1, 3096, (1, 1, 1), None), ("k_huff_hist2", 3, 8 * KB, (24, 1, 1), (1, 1, 1))),
    "image_fres_3_parts_n12": (("k_huff_hist2", 1, 3096, (1, 12, 1), None), ("k_huff_hist2", 3, 8 * KB, (24, 12, 1), (1, 12, 1))),
    "image_fres_2_parts": (("k_huff_hist2", 1, 3096, (1, 20, 1), None), ("k_huff_hist2", 2, 16 * KB, (16, 20, 1), (1, 20, 1))),
    "image_fres_no_parts": (("k_huff_hist2", 1, 3096, (1, 40, 1), None), ("k_huff_hist2", 1, 24576, (8, 40, 1), (1, 40, 1))),
    "image_1080p_lres_12_parts": (("k_huff_hist2", 12, 8 * KB, (12, 1, 1), None),
                                  ("k_huff_hist2", 3, 16 * KB, (405, 1, 1), (1, 1, 1))),
    "image_4096_gray_lres_parts": (("k_huff_hist2", 33, 8 * KB, (33, 1, 1), None),
                                   ("k_huff_hist2", 1, 32 * KB, (512, 1, 1), (2, 1, 1))),
    "image_lres_2_parts_fres_teams": (("k_huff_hist2", 2, 16 * KB, (2, 600, 1), None),
                                      ("k_huff_hist4", 1, 8 * KB, (16, 600, 1), (1, 600, 1))),
    "image_generic": (("k_huff_hist", 1, 3096, (1, 2, 1), None), ("k_huff_hist", 1, 24576, (8, 2, 1), (1, 2, 1))),
}


def summary(s):
    return (s.hist, s.nsub, s.sub_size, s.grid, s.stale)


def test_shape_matrix_mirror():
    """The mirror maps every matrix entry to the shape listed, and the matrix reaches every kernel pair, part counts
    of 1, 2, 3, 9, 12, 33 and 64, a short last part and warp teams with a partial last CTA."""
    got = {}
    for name, kind, args, opt in MATRIX:
        s = shape_of(kind, args, opt)
        got[name] = summary(s) if kind == "stage" else tuple(summary(c) for c in s)
    assert got == MATRIX_SHAPES
    shapes = [shape_of(k, a, o) for _, k, a, o in MATRIX]
    flat = [c for s in shapes for c in (s if isinstance(s, tuple) and isinstance(s[0], Shape) else (s,))]
    assert {c.hist for c in flat} == {"k_huff_hist", "k_huff_hist2", "k_huff_hist4"}
    assert {1, 2, 3, 9, 12, 33, 64} <= {c.nsub for c in flat}
    assert 70000 % (8 * KB) and 131 % TEAM_WARPS  # a short last part; a partial last CTA of warp teams
    assert stage_shape(37, 131 * 1000, 1000).hist == "k_huff_hist4" and 37 * 131 >= WAVE > 36 * 131
    # the low-res chunk of a 1024x1024 gray image is just over 16 KiB: parts from 1 to 1183 images, none from 1184
    assert image_geom(1024, 1024, 1)[0] > 16 * KB
    assert image_shapes(1183, 1024, 1024, 1)[0].nsub == 2 and image_shapes(1184, 1024, 1024, 1)[0].nsub == 1
    assert image_shapes(591, 1024, 1024, 1)[0].nsub == 3


# ---------------------------------------------------------------------------------------------
# CPU model of the tokens, the part bit counts and the stale padding
# ---------------------------------------------------------------------------------------------
def run_symbols(z):
    """Symbol of the last token of runs of z >= 1 zeros (after the maximal tokens)."""
    return np.select([z == 1, z == 2, z <= 6, z <= 22, z <= 278], [0, 256, 257, 258, 259], 260)


def runs(data, seg_size):
    """Zero runs of every segment: (start, length, position of the item that ends it or -1 at the segment end)."""
    p = np.flatnonzero(data)
    s = p // seg_size
    prev = np.r_[-1, p[:-1]][: p.size]
    first = np.r_[True, s[1:] != s[:-1]][: p.size]
    prev = np.where(first, s * seg_size - 1, prev)
    gap = p - prev - 1
    nseg = data.size // seg_size
    last = np.full(nseg, -1, np.int64)
    np.maximum.at(last, s, p - s * seg_size)
    seg_ids = np.arange(nseg)
    tail = seg_size - 1 - last
    starts = np.r_[p[gap > 0] - gap[gap > 0], (seg_ids * seg_size + last + 1)[tail > 0]]
    lens = np.r_[gap[gap > 0], tail[tail > 0]]
    items = np.r_[p[gap > 0], np.full(int((tail > 0).sum()), -1)]
    return starts.astype(np.int64), lens.astype(np.int64), items.astype(np.int64)


def part_hists(data, seg_size, sub_size):
    """[nseg][nsub][261] token histograms of the parts: a run counts in the part of the item that ends it, or in
    the last part when it is still open at the segment end; maximal tokens are cut greedily from its start."""
    nseg, nsub = data.size // seg_size, -(-seg_size // sub_size)
    H = np.zeros((nseg * nsub, 261), np.int64)
    p = np.flatnonzero(data)
    s = p // seg_size
    row = s * nsub + (p - s * seg_size) // sub_size
    np.add.at(H, (row, data[p].astype(np.int64)), 1)
    st, ln, it = runs(data, seg_size)
    rrow = np.where(it >= 0, (it // seg_size) * nsub + (it % seg_size) // sub_size, (st // seg_size) * nsub + nsub - 1)
    np.add.at(H, (rrow, np.full(rrow.size, 260)), ln // MAX_RUN)
    rest = ln % MAX_RUN
    m = rest > 0
    np.add.at(H, (rrow[m], run_symbols(rest[m])), 1)
    return H.reshape(nseg, nsub, 261)


def code_lengths(port, data, bs):
    _, code, ln, _ = port.huff_tree(port.huff_histogram(data, bs))
    return code, ln.astype(np.int64)


def part_bits(port, data, bs, sub_size, ln=None):
    """[nseg][nsub] bits of every part: part histogram . (code length + extra bits)."""
    seg = bs if bs > 0 else data.size
    if ln is None:
        ln = code_lengths(port, data, bs)[1]
    return part_hists(data, seg, sub_size) @ (ln + EXTRA)


def oracle_segment_bytes(port, packed, data, bs):
    """Payload bytes of every segment of the oracle's stream (from its segment headers)."""
    tree_bytes = (port.huff_tree(port.huff_histogram(data, bs))[0] + 7) // 8
    if bs <= 0:
        return [len(packed) - tree_bytes], [tree_bytes]
    sizes, at, pos = [], [], tree_bytes
    for _ in range(data.size // bs):
        sz, hl = packed[pos] | packed[pos + 1] << 8, 2
        if sz & 0x8000:
            sz, hl = (sz & 0x7FFF) | (packed[pos + 2] | packed[pos + 3] << 8) << 15, 4
        sizes.append(sz)
        at.append(pos + hl)
        pos += hl + sz
    assert pos == len(packed)
    return sizes, at


def stale_sources(bits):
    """For every segment, the (source segment, first bit, end bit) spans of its padding bits: the most recent earlier
    segment longer than the next padding bit (k_huff_stale's rule), through a stack of candidate segments."""
    out, stack = [], []  # stack: segments no later segment is at least as long as, lengths decreasing upwards
    for b, lo in enumerate(int(x) for x in bits):
        hi, spans = (lo + 7) & ~7, []
        for e in reversed(stack):
            if lo >= hi:
                break
            if bits[e] > lo:
                upto = min(int(bits[e]), hi)
                spans.append((e, lo, upto))
                lo = upto
        out.append(spans)
        while stack and bits[stack[-1]] <= bits[b]:
            stack.pop()
        stack.append(b)
    return out


def piece_stats(data, seg_size, sub_size):
    """Per 8 KiB piece of every part (pieces start at the part start): (segment, part, piece index in the part,
    items, zeros carried in, position of its first item or -1)."""
    out = []
    p = np.flatnonzero(data)
    for s in range(data.size // seg_size):
        for q0 in range(0, seg_size, sub_size):
            for k, b in enumerate(range(q0, min(q0 + sub_size, seg_size), PIECE)):
                a0, a1 = s * seg_size + b, s * seg_size + min(b + PIECE, q0 + sub_size, seg_size)
                i0, i1 = np.searchsorted(p, a0), np.searchsorted(p, a1)
                before = p[i0 - 1] if i0 > 0 and p[i0 - 1] >= s * seg_size else s * seg_size - 1
                out.append((s, q0 // sub_size, k, int(i1 - i0), int(a0 - 1 - before), int(p[i0] - a0) if i1 > i0 else -1))
    return out


# ---------------------------------------------------------------------------------------------
# corpus: each stream is built for one seam, stated (and checked on the CPU) next to its builder
# ---------------------------------------------------------------------------------------------
def background(rng, size, density=0.25):
    """Sparse small literals, like quantised coefficient planes."""
    d = np.minimum(rng.geometric(0.35, size), 255).astype(np.uint8)
    d[rng.random(size) >= density] = 0
    return d


def set_items(rng, data, a, b, count):
    """Exactly `count` non-zero bytes in data[a:b]."""
    data[a:b] = 0
    data[a + rng.choice(b - a, count, replace=False)] = rng.integers(1, 9, count).astype(np.uint8)


FIB = [1, 1]
while len(FIB) < 40:
    FIB.append(FIB[-1] + FIB[-2])


def fibonacci_literals(nlit):
    """Literals nlit .. 1 with counts 1, 2, 3, 5, ... (Fibonacci): the deepest tree nlit symbols can give."""
    return np.concatenate([np.full(c, nlit - k, np.uint8) for k, c in enumerate(FIB[1:1 + nlit])])


P16 = 16 * KB  # part size of a 1 MiB unframed stream at n = 1
P64 = 64 * KB  # part size of a 4 MiB unframed stream at n = 1


def build_lookback():
    rng = np.random.default_rng(1)
    d = background(rng, MIB)
    d[5 * P16 + 1000: 8 * P16 + 2000] = 0  # 50 152 zeros from part 5 to the item in part 8
    d[8 * P16 + 2000] = 3
    d[20 * P16 - 1], d[20 * P16: 20 * P16 + 300], d[20 * P16 + 300] = 4, 0, 5  # a run that starts at a part start
    d[30 * P16 - 1], d[30 * P16] = 6, 7  # items at p0 - 1 and p0
    return d, 0, 1


def props_lookback(port, d, bs, sh):
    st, ln, it = runs(d, d.size)
    far = (it >= 0) & (it // sh.sub_size - st // sh.sub_size >= 2) & (ln >= 40000)
    assert far.any() and ln[far].max() > 20 * LOOKBACK  # the look-back takes many windows
    assert ((st % sh.sub_size == 0) & (st > 0) & (it >= 0)).any()
    p0 = 30 * sh.sub_size
    assert d[p0 - 1] and d[p0]


def build_greedy_cuts():
    rng = np.random.default_rng(2)
    d = background(rng, MIB)
    for k, L in enumerate((16661, 16662, 16663, 33324, 33325)):
        s = (3 * k + 2) * P16 + 10000
        d[s - 1], d[s: s + L], d[s + L] = 2, 0, 9
    return d, 0, 1


def props_greedy_cuts(port, d, bs, sh):
    st, ln, it = runs(d, d.size)
    for L in (16661, 16662, 16663, 33324, 33325):
        k = np.flatnonzero(ln == L)
        assert k.size == 1 and it[k[0]] >= 0, L
        # the greedy cuts start where the run starts, in another part than the item the run counts with
        assert st[k[0]] // sh.sub_size != it[k[0]] // sh.sub_size, L


def build_empty_tail():
    rng = np.random.default_rng(3)
    d = background(rng, MIB)
    d[61 * P16 + 5000:] = 0  # the last two parts all zero: a run from part 61 ends at the segment end
    return d, 0, 1


def props_empty_tail(port, d, bs, sh):
    pb = part_bits(port, d, bs, sh.sub_size)[0]
    assert sh.nsub == 64 and not d[62 * sh.sub_size:].any() and pb[62] == 0 and pb[63] > 0
    H = part_hists(d, d.size, sh.sub_size)[0]
    run = d.size - 1 - np.flatnonzero(d)[-1]
    assert run > 2 * sh.sub_size and run % MAX_RUN >= 279  # (the rest of the run is a symbol-260 token too)
    assert H[63].sum() == H[63, 260] == run // MAX_RUN + 1


def build_byte_seams():
    """Parts ending mid-byte and on a byte boundary, and an all-zero (zero-bit) part 40 between parts 39 and 41
    that OR the same byte; the background is reseeded until part 40 starts mid-byte."""
    for seed in range(100):
        rng = np.random.default_rng(100 + seed)
        d = background(rng, MIB)
        d[40 * P16 - 3: 41 * P16 + 7] = 0
        d[41 * P16 + 7] = 1
        _, ln = code_lengths(PORT[0], d, 0)
        start = np.r_[0, np.cumsum(part_bits(PORT[0], d, 0, P16, ln)[0])]
        if start[40] % 8 and (start[1:64] % 8 == 0).any():
            return d, 0, 1
    raise AssertionError("no seed gives the seams")


def props_byte_seams(port, d, bs, sh):
    pb = part_bits(port, d, bs, sh.sub_size)[0]
    start = np.r_[0, np.cumsum(pb)]
    assert pb[40] == 0 and start[40] % 8 and start[41] == start[40]
    assert (start[1:sh.nsub] % 8 == 0).any() and (start[1:sh.nsub] % 8 != 0).any()


def build_pieces():
    rng = np.random.default_rng(4)
    d = background(rng, 4 * MIB, 0.1)
    for part, piece, count in ((2, 0, 2048), (4, 0, 2049), (6, 3, 2048), (8, 3, 2049)):
        a = part * P64 + piece * PIECE
        set_items(rng, d, a, a + PIECE, count)
    # first gaps of 16 662 zeros or more with zeros carried in: 16 776, exactly 2 x 16 662, and one carried into
    # a part from the part before it (the look-back)
    for part, z0, z1, after in ((10, 1 * PIECE + 8000, 4 * PIECE + 200, 7), (12, 8092, 5 * PIECE + 456, 8),
                                (14, -2 * PIECE, 500, 9)):
        a = part * P64
        d[a + z0 - 1], d[a + z0: a + z1], d[a + z1] = 3, 0, after
    return d, 0, 1


def props_pieces(port, d, bs, sh):
    assert sh.sub_size == P64 and sh.sub_size // PIECE == 8
    ps = piece_stats(d, d.size, sh.sub_size)
    last = sh.sub_size // PIECE - 1
    for count in (ITEM_CAP, ITEM_CAP + 1):
        assert any(k == 0 and c == count for _, _, k, c, _, _ in ps), count
        assert any(0 < k < last and c == count for _, _, k, c, _, _ in ps), count
    gap0 = [(k, zin, zin + f) for _, _, k, c, zin, f in ps if c and zin]
    assert any(g > MAX_RUN and g % MAX_RUN for _, _, g in gap0)
    assert any(g == 2 * MAX_RUN for _, _, g in gap0)
    assert any(k == 0 and zin >= 2 * PIECE and g >= MAX_RUN for k, zin, g in gap0)


TEAM_SEG = 24576


def build_team_caps():
    rng = np.random.default_rng(5)
    d = background(rng, 40 * TEAM_SEG, 0.1)
    cap = 3 * ITEM_CAP  # pieces_per_part x kItemCap of a 24 576-byte segment
    set_items(rng, d, 3 * TEAM_SEG, 4 * TEAM_SEG, cap)
    set_items(rng, d, 4 * TEAM_SEG, 5 * TEAM_SEG, cap + 1)
    set_items(rng, d, 5 * TEAM_SEG, 6 * TEAM_SEG - 1, cap - 1)
    d[6 * TEAM_SEG - 1] = 4  # exactly the capacity, the last item in the last byte
    d[7 * TEAM_SEG: 8 * TEAM_SEG] = 0
    return d, TEAM_SEG, 8


def props_team_caps(port, d, bs, sh):
    t = stage_shape(8, d.size, bs, teams=2)
    assert t.hist == "k_huff_hist4" and t.pieces_per_part == 3
    counts = (d.reshape(-1, bs) != 0).sum(1)
    assert {3 * ITEM_CAP, 3 * ITEM_CAP + 1} <= set(counts.tolist()) and d[6 * bs - 1]


RUN_SEG = 100000


def build_team_u16_runs():
    rng = np.random.default_rng(6)
    d = background(rng, 12 * RUN_SEG, 0.05)
    for s, L in ((1, 65535), (2, 65536), (4, 65535), (5, 65536), (7, 65535 + MAX_RUN)):
        a = s * RUN_SEG + 1000
        d[a - 1], d[a: a + L], d[a + L] = 1, 0, 2
    d[9 * RUN_SEG - 65535: 9 * RUN_SEG] = 0  # a run of exactly 65 535 zeros at a segment end
    d[9 * RUN_SEG - 65536] = 3
    d[11 * RUN_SEG - 65536: 11 * RUN_SEG] = 0
    d[11 * RUN_SEG - 65537] = 3
    return d, RUN_SEG, 25


def props_team_u16_runs(port, d, bs, sh):
    assert stage_shape(25, d.size, bs, teams=2).hist == "k_huff_hist4"
    st, ln, it = runs(d, bs)
    for L in (65535, 65536):
        assert ((ln == L) & (it >= 0)).any() and ((ln == L) & (it < 0)).any(), L


def build_odd(seg, nseg):
    def build():
        rng = np.random.default_rng(seg)
        return background(rng, seg * nseg, 0.3), seg, 1
    return build


def props_odd(port, d, bs, sh):
    n = [n for n, opt, odd in corpus_configs(d.size, bs, 1) if opt == "teams" and odd]
    assert bs % 16 and len(n) == 1 and stage_shape(n[0], d.size, bs, teams=2).hist == "k_huff_hist4"


LONG_SIZE = 14930350  # Fibonacci counts 1, 2, 3, ..., F(34) over 33 literals
LONG_SEG = 298607  # 50 segments of it (an odd segment size)


def build_long_codes(bs):
    def build():
        d = fibonacci_literals(33)
        np.random.default_rng(7).shuffle(d)
        return d, bs, 1
    return build


def props_long_codes(port, d, bs, sh):
    assert d.size == LONG_SIZE
    _, ln = code_lengths(port, d, bs)
    assert ln.max() == 32 and set(range(1, 33)) <= set(ln.tolist())
    if bs == 0:
        assert sh.nsub == 63 and sh.sub_size == 237568


def build_long_runs():
    """The 33-symbol Fibonacci tree with its two rarest symbols being zero runs (one of 300 zeros: run symbol 260,
    two of 100: symbol 259), each in front of one of the rarest literals: items of run code + 14 or 8 extra bits +
    literal code, over 64 bits."""
    counts = FIB[1:34]
    lits = np.concatenate([np.full(c, 31 - k, np.uint8) for k, c in enumerate(counts[2:])])
    rng = np.random.default_rng(8)
    rng.shuffle(lits)
    where = np.flatnonzero(lits == 31)[:3]  # (literal 31 is the rarest one)
    pieces, at = [], 0
    for w, z in zip(where, (300, 100, 100)):
        pieces += [lits[at:w], np.zeros(z, np.uint8)]
        at = w
    pieces.append(lits[at:])
    d = np.concatenate(pieces)
    return d, 0, 1


def props_long_runs(port, d, bs, sh):
    _, ln = code_lengths(port, d, bs)
    assert ln.max() == 32 and ln[260] >= 31 and ln[259] >= 30
    st, rl, it = runs(d, d.size)
    assert rl.size == 3 and (it >= 0).all()
    bits = ln[run_symbols(rl)] + EXTRA[run_symbols(rl)] + ln[d[it]]
    assert bits.max() > 64


STALE_N, STALE_SEG = 3000, 64


def stale_base(rng):
    d = np.zeros((STALE_N, STALE_SEG), np.uint8)
    d[0] = rng.integers(1, 256, STALE_SEG)
    d[1:, 5], d[1:, 40] = 1, 2
    return d


EDGE = {"edge_1024": 1280 - STALE_WINDOW, "edge_1025": 1280 - STALE_WINDOW - 1}  # a long segment at / just before
# the window start of the CTA of segments 1280 .. 1535


def build_stale(variant):
    """3000 framed 64-byte segments: segment 0 random literals, the others zero but for bytes 5 and 40 (29 bits
    each).  edge_*: a second long segment at EDGE; two_sources: segment 1000 a bit or two longer than the short ones
    (the first of the byte changes that gives that).  Seeds are tried until the padding bits of the long segments
    are not all zero and differ from each other, so that a wrong source shows."""
    def build():
        for seed in range(9, 100):
            rng = np.random.default_rng(seed)
            d = stale_base(rng)
            if variant in EDGE:
                d[EDGE[variant]] = rng.integers(1, 256, STALE_SEG)
            if variant == "two_sources":
                for at, v in ((41, 1), (41, 2), (6, 1), (6, 2), (39, 1), (39, 2), (4, 1), (4, 2)):
                    t = d.copy()
                    t[1000, at] = v
                    pb = part_bits(PORT[0], t.reshape(-1), STALE_SEG, STALE_SEG)[:, 0]
                    if pb[1000] in (30, 31) and pb[1] == 29:
                        d = t
                        break
            flat = d.reshape(-1)
            packed = np.frombuffer(PORT[0].huff_compress(flat, STALE_SEG), np.uint8)
            _, at = oracle_segment_bytes(PORT[0], packed.tobytes(), flat, STALE_SEG)
            pads = {int(packed[at[e] + 3]) & 0xE0 for e in (0, EDGE.get(variant, 0))}
            if 0 not in pads and len(pads) == 1 + (variant in EDGE):
                return flat, STALE_SEG, 1
        raise AssertionError("no seed")
    return build


def props_stale(variant):
    def props(port, d, bs, sh):
        pb = part_bits(port, d, bs, bs)[:, 0]
        packed = np.frombuffer(port.huff_compress(d, bs), np.uint8)
        _, at = oracle_segment_bytes(port, packed.tobytes(), d, bs)
        src = stale_sources(pb)
        short = np.flatnonzero(pb == 29)
        assert pb[0] > 32 and short.size >= STALE_N - 2
        cta = range(1280, 1536)
        if variant == "plain":  # every short segment's padding from segment 0: last byte 0xC0
            assert short.size == STALE_N - 1 and all(src[b] == [(0, 29, 32)] for b in short)
            pad = packed[at[0] + 3] & 0xE0  # (not zero: a padding left at zero shows)
            assert pad and all(packed[at[b] + 3] == pad | (packed[at[1] + 3] & 0x1F) for b in short)
            # from segment 1280 on, more than kStaleWindow segments before the CTA's first one
            assert all(0 < (b // 256) * 256 - STALE_WINDOW for b in range(1280, STALE_N)) and 1280 % 256 == 0
        elif variant in EDGE:
            e = EDGE[variant]
            assert all(src[b] == [(e, 29, 32)] for b in cta)
            assert (packed[at[e] + 3] ^ packed[at[0] + 3]) & 0xE0 and packed[at[e] + 3] & 0xE0  # a wrong source shows
        else:  # bits [29, L) from segment 1000 (inside the window), the rest from segment 0 (outside it)
            L = int(pb[1000])
            assert L in (30, 31) and all(src[b] == [(1000, 29, L), (0, L, 32)] for b in cta)
            assert 1000 >= 1280 - STALE_WINDOW
    return props


def build_single(value):
    def build():
        return np.full(MIB, value, np.uint8), 0, 1
    return build


def props_single(port, d, bs, sh):
    _, ln = code_lengths(port, d, bs)
    assert (ln > 0).sum() == 1 and sh.nsub == 64
    pb = part_bits(port, d, bs, sh.sub_size)[0]
    if not d.any():  # every run token from the last part
        assert (pb[:-1] == 0).all() and pb[-1] > 0


# name -> (builder, property check); a builder returns (data, block size, batch size of the shape the properties
# are stated for)
CORPUS = {
    "lookback": (build_lookback, props_lookback),
    "greedy_cuts": (build_greedy_cuts, props_greedy_cuts),
    "empty_tail": (build_empty_tail, props_empty_tail),
    "byte_seams": (build_byte_seams, props_byte_seams),
    "pieces": (build_pieces, props_pieces),
    "team_caps": (build_team_caps, props_team_caps),
    "team_u16_runs": (build_team_u16_runs, props_team_u16_runs),
    "odd_33": (build_odd(33, 300), props_odd),
    "odd_1001": (build_odd(1001, 200), props_odd),
    "odd_24577": (build_odd(24577, 12), props_odd),
    "long_codes_unframed": (build_long_codes(0), props_long_codes),
    "long_codes_framed": (build_long_codes(LONG_SEG), props_long_codes),
    "long_codes_runs": (build_long_runs, props_long_runs),
    "stale_window": (build_stale("plain"), props_stale("plain")),
    "stale_edge_1024": (build_stale("edge_1024"), props_stale("edge_1024")),
    "stale_edge_1025": (build_stale("edge_1025"), props_stale("edge_1025")),
    "stale_two_sources": (build_stale("two_sources"), props_stale("two_sources")),
    "single_literal": (build_single(7), props_single),
    "all_zero": (build_single(0), props_single),
}

PORT = []  # the oracle port, for the builders that search seeds
_BUILT = {}


def corpus(port, name):
    if not PORT:
        PORT.append(port)
    if name not in _BUILT:
        _BUILT[name] = CORPUS[name][0]()
    return _BUILT[name]


BATCH_BYTES = 96 * MIB  # input bytes of one corpus call


def corpus_configs(size, bs, n0):
    """(n, context, odd input stride) of every shape a stream reaches: the batch its properties are stated for,
    the first batch without parts (a CTA per segment, and warp teams for framed streams), the first-generation
    pair and both with the item lists off.  The warp-team calls read rows at an odd stride."""
    nseg = size // (bs if bs > 0 else size)
    n_np = next((n for n in (1, 2, 3, 4, 6, 8, 12, 25, 40, 80, 160, 300) if stage_shape(n, size, bs).nsub == 1
                 and n * size <= BATCH_BYTES), None)
    cfg = [(n0, "default", False), (1, "generic", False), (n0, "nolists", False)]
    if n_np and nseg > 1:
        cfg += [(n_np, "ctas", False), (n_np, "teams", True), (n_np, "nolists_teams", False)]
    elif nseg == 1:  # another part count
        n1 = next((n for n in (3, 20, 600) if n * size <= BATCH_BYTES and stage_shape(n, size, bs).nsub != stage_shape(n0, size, bs).nsub), None)
        cfg += [(n1, "default", False)] if n1 else []
    seen, out = set(), []
    for n, opt, odd in cfg:
        key = (n, opt)
        if key not in seen:
            seen.add(key)
            out.append((n, opt, odd))
    return out


@pytest.mark.parametrize("name", list(CORPUS))
def test_corpus_properties(port, name):
    """Each stream has the seam it is built for, at the shape it is stated for (CPU only)."""
    d, bs, n0 = corpus(port, name)
    CORPUS[name][1](port, d, bs, stage_shape(n0, d.size, bs))
    assert len(port.huff_compress(d, bs)) > 0


@pytest.mark.parametrize("name", list(CORPUS))
def test_part_bits_model(port, name):
    """Per segment, the parts' histograms sum to the oracle's segment histogram, and their bits to the payload of
    the oracle's segment, in every shape the stream reaches (CPU only)."""
    d, bs, n0 = corpus(port, name)
    seg = bs if bs > 0 else d.size
    _, ln = code_lengths(port, d, bs)
    packed = port.huff_compress(d, bs)
    seg_bytes, _ = oracle_segment_bytes(port, packed, d, bs)
    subs = {stage_shape(n, d.size, bs, *OPTIONS[o][:2]).sub_size for n, o, _ in corpus_configs(d.size, bs, n0)}
    whole = part_hists(d, seg, seg)[:, 0]
    for s in range(min(d.size // seg, 64)):
        assert np.array_equal(whole[s], port.huff_histogram(d[s * seg: (s + 1) * seg], 0).astype(np.int64)), s
    for sub in subs:
        H = part_hists(d, seg, sub)
        assert np.array_equal(H.sum(1), whole), sub
        bits = (H @ (ln + EXTRA)).sum(1)
        assert [int(b + 7) // 8 for b in bits] == seg_bytes, sub


def test_stale_model_on_the_oracle(port):
    """stale_sources is the oracle's padding rule: rebuilding every padded byte of a framed stream from its sources'
    bytes gives the oracle's bytes (CPU only)."""
    for name in ("stale_window", "stale_edge_1025", "stale_two_sources", "odd_1001"):
        d, bs, _ = corpus(port, name)
        packed = np.frombuffer(port.huff_compress(d, bs), np.uint8)
        _, at = oracle_segment_bytes(port, packed.tobytes(), d, bs)
        bits = part_bits(port, d, bs, bs)[:, 0]
        for b, spans in enumerate(stale_sources(bits)):
            if bits[b] % 8 == 0:
                continue
            byte = int(bits[b]) >> 3
            want = 0
            for e, lo, upto in spans:
                mask = ((1 << (upto - 8 * byte)) - 1) & ~((1 << (lo - 8 * byte)) - 1)
                want |= int(packed[at[e] + byte]) & mask
            own = int(packed[at[b] + byte]) & ((1 << (int(bits[b]) - 8 * byte)) - 1)
            assert packed[at[b] + byte] == own | want, (name, b)


# ---------------------------------------------------------------------------------------------
# GPU helpers: contexts, raw stage calls, status, traces
# ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ctxs():
    torch = pytest.importorskip("torch")
    import himg_b200

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    cs = {}
    for name, (g, t, l) in OPTIONS.items():
        c = himg_b200.Context(0)
        c.set_option("force_generic", int(g))
        c.set_option("huff_warp_teams", t)
        c.set_option("item_lists", int(l))
        cs[name] = c
    yield cs
    for c in cs.values():
        c.close()


def status_ok(ctx):
    """The device error flag after a coding call (read = clear): OK, or raises."""
    ctx.encode_status()


def status_of(ctx):
    import himg_b200

    try:
        ctx.encode_status()
    except himg_b200.HimgError as e:
        return e.code
    return OK


def odd_stride(size):
    """A row stride >= size that is 3 (mod 16)."""
    return size + (3 - size) % 16


def device_rows(data, n, odd=False):
    """n copies of data on the device; with odd, rows of a wider tensor (an odd row stride)."""
    import torch

    base = torch.from_numpy(np.ascontiguousarray(data)).cuda()
    if not odd:
        return base.unsqueeze(0).repeat(n, 1)
    buf = torch.empty((n, data.size + 3), dtype=torch.uint8, device="cuda")
    buf[:, : data.size] = base
    return buf[:, : data.size]


def compress(ctx, x, bs, stride=None):
    """himgcu_stage_huff_compress of the rows of x into a sentinel-filled [n][stride] buffer (stride 3 mod 16 by
    default).  Returns (out [n][stride] device tensor, sizes [n] int64 numpy)."""
    import torch

    n, in_size = x.shape
    stride = stride or odd_stride(2 * in_size + 4096)
    flat = torch.full((n * stride + 64,), SENTINEL, dtype=torch.uint8, device="cuda")
    sizes = torch.full((n,), -1, dtype=torch.int32, device="cuda")
    ctx._bind(x, flat, sizes, rows_ok=True)
    ctx._check(ctx.lib.himgcu_stage_huff_compress(ctx.h, x.data_ptr(), x.stride(0), n, in_size, bs, flat.data_ptr(), stride,
                                                  sizes.data_ptr()))
    torch.cuda.synchronize()
    assert (flat[n * stride:] == SENTINEL).all(), "bytes written past the last row"
    return flat[: n * stride].view(n, stride), sizes.cpu().numpy().astype(np.int64)


def check_rows(out, sizes, wants, what):
    """Row i of out holds wants[i] (bytes, or None: not coded, the whole row left at the sentinel), then the
    sentinel to the end of the row.  Compared on the device."""
    import torch

    cache = {}
    for i, w in enumerate(wants):
        if w is None:
            assert sizes[i] == 0, f"{what}, item {i}: size {sizes[i]}, expected 0"
            assert bool((out[i] == SENTINEL).all()), f"{what}, item {i}: a row that is not coded was written"
            continue
        size, want_size = int(sizes[i]), len(w)
        assert size == want_size, f"{what}, item {i}: size {size} vs {want_size}"
        if id(w) not in cache:
            cache[id(w)] = torch.from_numpy(np.frombuffer(w, np.uint8).copy()).cuda()
        row = out[i]
        if not bool((row[: len(w)] == cache[id(w)]).all()):
            got = row[: len(w)].cpu().numpy()
            d = np.flatnonzero(got != np.frombuffer(w, np.uint8))
            pytest.fail(f"{what}, item {i}: {d.size} bytes differ, first at {d[0]} of {len(w)}")
        tail = row[len(w):]
        assert bool((tail == SENTINEL).all()), f"{what}, item {i}: bytes behind the stream written"


def code_and_check(ctx, port, data, bs, n, what, odd=False, want=None):
    want = want if want is not None else port.huff_compress(data, bs)
    out, sizes = compress(ctx, device_rows(data, n, odd), bs)
    status_ok(ctx)
    check_rows(out, sizes, [want] * n, what)


def traced_launches(fn):
    """(kernel, grid, block) of every histogram, pack and stale launch of fn(), from a torch.profiler trace."""
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
    for e in sorted((e for e in events if e.get("cat") == "kernel"), key=lambda e: e.get("ts", 0)):
        m = re.search(r"(k_huff_(?:hist\d?|pack\d?|stale))(?=[<(])", e.get("name", ""))
        if m:
            a = e.get("args", {})
            out.append((m.group(1), tuple(a.get("grid", ())), tuple(a.get("block", ()))))
    return out


# ---------------------------------------------------------------------------------------------
# GPU tests
# ---------------------------------------------------------------------------------------------
def natural(port, size, seed):
    """FRES planes of a synthetic image, repeated to size bytes."""
    img = port.synth(1024, 64, 3, seed, 9)
    cm = port.rgb_to_ycbcr(img)
    return np.resize(port.fullres_planes(cm, port.lowres_sample(cm), 50, True), size)


STAGE_MATRIX = [m for m in MATRIX if m[1] == "stage"]
IMAGE_MATRIX = [m for m in MATRIX if m[1] == "image"]


@pytest.mark.gpu
@pytest.mark.parametrize("entry", STAGE_MATRIX, ids=[m[0] for m in STAGE_MATRIX])
def test_stage_shape_matrix(ctxs, port, entry):
    """Each stage entry launches the kernels, grids and blocks the mirror names, and codes four distinct streams
    (repeated over the batch) as the oracle does."""
    import torch

    name, _, (n, in_size, bs), opt = entry
    datas = [natural(port, in_size, s) for s in range(1, 1 + min(n, 4))]
    wants = [port.huff_compress(d, bs) for d in datas]
    x = torch.from_numpy(np.stack(datas)).cuda()[torch.arange(n) % len(datas)]
    ctx = ctxs[opt]
    res = {}
    got = traced_launches(lambda: res.update(r=compress(ctx, x, bs)))
    status_ok(ctx)
    assert got == launches([shape_of("stage", (n, in_size, bs), opt)]), f"{name}: launches {got}"
    check_rows(*res["r"], [wants[i % len(datas)] for i in range(n)], name)


def image_batch(port, n, w, h, nch):
    """n images on the device (at most 8 distinct ones, repeated) and the indices of the distinct ones."""
    import torch

    k = min(n, 8)
    imgs = np.stack([port.synth(w, h, nch, 10 + s, 6 + 9 * s) for s in range(k)])
    return torch.from_numpy(imgs).cuda()[torch.arange(n) % k], imgs


@pytest.mark.gpu
@pytest.mark.parametrize("entry", IMAGE_MATRIX, ids=[m[0] for m in IMAGE_MATRIX])
def test_image_shape_matrix(ctxs, port, entry):
    """encode_batch into a sentinel-filled out= with a row stride of 3 (mod 16): the launches the mirror names for
    both chunks, every distinct image the oracle's stream, every repeat equal to it, the sentinel behind each."""
    import torch

    name, _, (n, w, h, nch), opt = entry
    ctx = ctxs[opt]
    lres = int(ctx.lib.himgcu_lres_size(w, h, nch))
    assert lres == image_geom(w, h, nch)[0]
    px, imgs = image_batch(port, n, w, h, nch)
    stride = odd_stride(int(ctx.lib.himgcu_encode_bound(w, h, nch)) + 16)
    flat = torch.full((n * stride + 64,), SENTINEL, dtype=torch.uint8, device="cuda")
    out = flat[: n * stride].view(n, stride)
    res = {}
    got = traced_launches(lambda: res.update(r=ctx.encode_batch(px, 50, True, out=out)))
    status_ok(ctx)
    assert got == launches(shape_of("image", (n, w, h, nch), opt)), f"{name}: launches {got}"
    assert bool((flat[n * stride:] == SENTINEL).all())
    sizes = res["r"][1].cpu().numpy().astype(np.int64)
    wants = [port.encode(im, 50, True) for im in imgs]
    check_rows(out, sizes, [wants[i % len(wants)] for i in range(n)], name)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CORPUS))
def test_corpus_across_shapes(ctxs, port, name):
    """Every corpus stream, copied over the batch, is the oracle's stream in every shape it reaches."""
    d, bs, n0 = corpus(port, name)
    want = port.huff_compress(d, bs)
    assert want
    for n, opt, odd in corpus_configs(d.size, bs, n0):
        code_and_check(ctxs[opt], port, d, bs, n, f"{name}, n={n} {opt}{' odd stride' if odd else ''}", odd, want)


@pytest.mark.gpu
def test_refused_33_bit_code(ctxs, port):
    """34 Fibonacci literals give a 33-bit code: the oracle refuses the stream, the middle item of a batch gets size 0
    and ERR_UNSUPPORTED with its row untouched, and its neighbours (one with 32-bit codes) are exact."""
    import torch

    refused = fibonacci_literals(34)
    rng = np.random.default_rng(12)
    rng.shuffle(refused)
    assert refused.size == 24157815 and port.huff_compress(refused, 0) == b""
    deep = np.where(refused == 34, 33, refused).astype(np.uint8)  # the two rarest literals merged: 32-bit codes
    assert code_lengths(port, deep, 0)[1].max() == 32
    other = background(rng, refused.size)
    x = torch.from_numpy(np.stack([deep, refused, other])).cuda()
    for opt in ("default", "generic"):
        ctx = ctxs[opt]
        out, sizes = compress(ctx, x, 0)
        assert status_of(ctx) == ERR_UNSUPPORTED, opt
        status_ok(ctx)  # (read = clear)
        check_rows(out, sizes, [port.huff_compress(deep, 0), None, port.huff_compress(other, 0)], f"33-bit code {opt}")


CAPACITY = [("unframed_parts", 100000, 0, "default"), ("framed_parts", 5 * 20000, 20000, "default"),
            ("teams", 13 * 4096, 4096, "teams"), ("generic", 3 * 20000, 20000, "generic")]


@pytest.mark.gpu
@pytest.mark.parametrize("what,in_size,bs,opt", CAPACITY, ids=[c[0] for c in CAPACITY])
def test_output_stride_only_some_items_fit(ctxs, port, what, in_size, bs, opt):
    """An out_stride (3 mod 16) between the packed sizes of the items: the ones that do not fit get size 0 and
    ERR_CAPACITY, their rows keep the sentinel, and their neighbours are exact."""
    import torch

    rng = np.random.default_rng(in_size)
    datas = [natural(port, in_size, 1), rng.integers(0, 256, in_size).astype(np.uint8), natural(port, in_size, 2),
             rng.integers(0, 256, in_size).astype(np.uint8)]
    wants = [port.huff_compress(d, bs) for d in datas]
    stride = odd_stride(max(len(wants[0]), len(wants[2])) + 5)
    assert len(wants[1]) > stride and len(wants[3]) > stride
    x = torch.from_numpy(np.stack(datas)).cuda()
    ctx = ctxs[opt]
    out, sizes = compress(ctx, x, bs, stride)
    assert status_of(ctx) == ERR_CAPACITY
    status_ok(ctx)
    check_rows(out, sizes, [wants[0], None, wants[2], None], what)


def test_reference_agrees(ref, port):
    """The oracle's streams of a sample of the corpus are the reference's."""
    for name in ("greedy_cuts", "byte_seams", "team_u16_runs", "odd_1001", "stale_edge_1025", "all_zero"):
        d, bs, _ = corpus(port, name)
        assert ref.huff_compress(d, bs) == port.huff_compress(d, bs), name
