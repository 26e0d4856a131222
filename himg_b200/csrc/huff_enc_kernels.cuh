// RLE + Huffman ENCODE kernels (reference: huffman_enc.cpp:98-363).
//
//   k_huff_hist2   zero-run tokenisation over a balanced item list + 261-bin histogram per segment
//                  (or per part of a segment)
//   k_huff_tree    one CTA per chunk: histogram total -> Huffman tree with the reference's exact
//                  tie-breaking -> (code,len) table + serialised tree
//   k_huff_layout  per item: segment bit lengths (histogram . code length), first bit of every part,
//                  prefix sum of (header + payload) sizes -> absolute byte offsets; container headers
//   k_huff_pack3   CTA per segment (or part): tokens built once in registers -> scan of bit totals ->
//                  word-wise accumulation into a shared-memory bit window -> bytes to the final position
//   k_huff_hist4 / k_huff_pack4 warp teams for framed chunks without parts: a warp per segment, one
//                  contiguous item list per segment, __syncwarp only
//   k_huff_hist / k_huff_pack   first-generation kernels (per-thread chunk walks): the force_generic path
//   k_huff_stale   the reference's uncleared scratch buffer leaks "stale" bits into the padding of
//                  every segment's last byte (SURVEY A.3 step 5); reproduced as a fix-up pass
//
// Tokenisation is "emit at run end": a thread owns the tokens that END inside its 32-byte chunk,
// so it only needs the number of zeros immediately preceding the chunk (one forward scan), and
// tokens stay in stream order.
#ifndef HIMG_B200_HUFF_ENC_KERNELS_CUH_
#define HIMG_B200_HUFF_ENC_KERNELS_CUH_

#include "common.cuh"

namespace himgcu {

constexpr int kHuffThreads = 512;
constexpr int kChunkBytes = 32;
constexpr int kPieceBytes = kHuffThreads * kChunkBytes;  // 16 KiB per CTA iteration
constexpr int kWinWords = 8192;                          // bit window: 32 KiB + 2 words of slack
constexpr int kWinBits = kWinWords * 32;

struct HuffGeom {
  int in_size;   // unpacked bytes per chunk
  int seg_size;  // bytes per segment (== in_size when the chunk is unframed)
  int nseg;
  unsigned long long in_stride;  // bytes between the chunks of consecutive items
  // A segment may be coded by `nsub` CTAs, each taking `sub_size` bytes (a multiple of the 8 KiB
  // piece): the segment stays ONE bit stream; the parts meet at arbitrary bit positions.  Used for
  // the single unframed low-res stream of large images when the batch alone cannot fill the GPU.
  int nsub;
  int sub_size;
};

// Mixed-geometry batch (encode): the chunk of item i belongs to an image of its own size, laid out with its own
// geometry at the start of a slot of the bounding geometry.  The kernels keep the bounding HuffGeom for the slot
// strides of every per-segment table (nseg, nsub) and take the item's own chunk geometry from mixed_chunk: the LRES
// chunk is one unframed segment of gi.lres_size bytes, the FRES chunk gi.rows segments of gi.seg bytes.  Mixed
// chunks have no parts (nsub = 1).  Segments past an item's own, and every segment of an image whose dims are out of
// bounds, are idle: the histogram pass writes zero rows for them and nothing reads or writes their bytes.
struct MixedHuff {
  MixedDims md;
  int fres;  // 0: the LRES chunk, 1: the FRES chunk
};
// Item `item`'s chunk geometry (hg: the bounding one on entry).  False when the image's dims are out of bounds.
__device__ __forceinline__ bool mixed_chunk(const MixedHuff &m, int item, HuffGeom &hg) {
  Geom gi;
  const bool ok = image_geom(m.md, item, gi);
  if (m.fres) {
    hg.seg_size = hg.sub_size = gi.seg;
    hg.nseg = gi.rows;
    hg.in_size = gi.rows * gi.seg;
  } else {
    hg.seg_size = hg.sub_size = hg.in_size = gi.lres_size;
    hg.nseg = 1;
  }
  return ok;
}

struct TreeOut {
  uint32_t code[kSyms];
  uint32_t hist[kSyms];
  uint8_t len[kSyms + 3];
  uint8_t tree[kTreeBytesMax];
  uint32_t tree_bits;
  uint32_t nleaves;
};

__device__ __forceinline__ int sym_extra_bits(int s) {
  return s < 257 ? 0 : (s == 257 ? 2 : (s == 258 ? 4 : (s == 259 ? 8 : 14)));
}

// ---- per-thread chunk of a segment ---------------------------------------------------------
// The 32 bytes of a thread are loaded with two coalesced 128-bit loads, parked in shared memory
// with a 9-word row stride (conflict-free for per-lane byte reads), and summarised as a bit mask
// of non-zero bytes.  Token walks then loop over the SET bits only (3 of 4 coefficient bytes are
// zero at quality 50), with one compact loop body instead of 32 unrolled byte positions.
constexpr int kRowWords = 9;

struct Chunk {
  const uint8_t *row;  // this thread's 36-byte row in shared memory
  uint32_t nz;         // bit p set <=> byte p is valid and non-zero
  int valid;           // number of valid bytes (0..32)
};

__device__ __forceinline__ uint32_t nonzero_nibble(uint32_t w) {
  // high bit of every byte set iff that byte is non-zero, then gather the four bits
  const uint32_t x = (((w & 0x7f7f7f7fu) + 0x7f7f7f7fu) | w) & 0x80808080u;
  return (((x >> 7) * 0x01020408u) >> 24) & 0xfu;
}

__device__ __forceinline__ void load_chunk(Chunk &c, uint32_t *rows, const uint8_t *__restrict__ seg,
                                           int seg_size, int off) {
  uint32_t w[8];
  c.valid = min(max(seg_size - off, 0), kChunkBytes);
#pragma unroll
  for (int k = 0; k < 8; ++k) w[k] = 0;
  if (c.valid == kChunkBytes && ((reinterpret_cast<uintptr_t>(seg + off)) & 15) == 0) {
    const uint4 a = __ldg(reinterpret_cast<const uint4 *>(seg + off));
    const uint4 b = __ldg(reinterpret_cast<const uint4 *>(seg + off) + 1);
    w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w;
    w[4] = b.x; w[5] = b.y; w[6] = b.z; w[7] = b.w;
  } else {
    for (int k = 0; k < c.valid; ++k) w[k >> 2] |= (uint32_t)seg[off + k] << (8 * (k & 3));
  }
  uint32_t *row = rows + threadIdx.x * kRowWords;
  uint32_t nz = 0;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    row[k] = w[k];
    nz |= nonzero_nibble(w[k]) << (4 * k);
  }
  c.row = reinterpret_cast<const uint8_t *>(row);
  c.nz = nz;  // bytes past `valid` were loaded as zero
}

// Zero-run summary of a chunk: low 31 bits = trailing zeros, bit 31 = "all zero" (an empty chunk
// is the identity).  combine(X earlier, Y later) is associative.
__device__ __forceinline__ uint32_t run_summary(const Chunk &c) {
  if (c.nz == 0) return (uint32_t)c.valid | 0x80000000u;
  return (uint32_t)(c.valid - 1 - (31 - __clz(c.nz)));
}
__device__ __forceinline__ uint32_t run_combine(uint32_t x, uint32_t y) {
  return (y & 0x80000000u) ? (((x & 0x7fffffffu) + (y & 0x7fffffffu)) | (x & 0x80000000u)) : y;
}

// Exclusive scan of run summaries over the block, seeded with the zeros carried in from earlier
// pieces.  Returns the number of zeros immediately preceding this thread's chunk; *carry_out is
// the trailing-zero count after the whole piece.  `ws` needs 17 words.
__device__ __forceinline__ uint32_t block_run_scan(uint32_t mine, uint32_t carry_in, uint32_t *ws, uint32_t *carry_out) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
  uint32_t inc = mine;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t t = __shfl_up_sync(0xffffffffu, inc, d);
    if (lane >= d) inc = run_combine(t, inc);
  }
  __syncthreads();
  if (lane == 31) ws[wid] = inc;
  __syncthreads();
  if (wid == 0) {
    uint32_t s = lane < nw ? ws[lane] : 0x80000000u;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, s, d);
      if (lane >= d) s = run_combine(t, s);
    }
    if (lane < nw) ws[lane] = s;
  }
  __syncthreads();
  uint32_t prev = __shfl_up_sync(0xffffffffu, inc, 1);
  if (lane == 0) prev = 0x80000000u;  // identity
  uint32_t ex = wid ? run_combine(ws[wid - 1], prev) : prev;
  const uint32_t seed = carry_in | 0x80000000u;
  ex = run_combine(seed, ex);
  *carry_out = run_combine(seed, ws[nw - 1]) & 0x7fffffffu;
  return ex & 0x7fffffffu;
}

// ---- token walk ------------------------------------------------------------------------------
template <class Sink>
__device__ __forceinline__ void emit_run(uint32_t z, Sink &s) {
  while (z >= (uint32_t)kMaxRun) {  // runs are cut greedily from their start (huffman_enc.cpp:111)
    s.tok(260, kMaxRun - 279, 14);
    z -= kMaxRun;
  }
  if (z == 0) return;
  if (z == 1) s.tok(0, 0, 0);
  else if (z == 2) s.tok(256, 0, 0);
  else if (z <= 6) s.tok(257, z - 3, 2);
  else if (z <= 22) s.tok(258, z - 7, 4);
  else if (z <= 278) s.tok(259, z - 23, 8);
  else s.tok(260, z - 279, 14);
}

// z_in: zeros immediately before the chunk; flush_end: the chunk holds the segment's last byte.
template <class Sink>
__device__ __forceinline__ void walk_chunk(const Chunk &c, uint32_t z_in, bool flush_end, Sink &s) {
  uint32_t mask = c.nz, carry = z_in;
  int prev = -1;
  while (mask) {
    const int p = __ffs(mask) - 1;
    mask &= mask - 1;
    const uint32_t z = (uint32_t)(p - prev - 1) + carry;
    carry = 0;
    prev = p;
    if (z) emit_run(z, s);
    s.tok((int)c.row[p], 0, 0);
  }
  if (flush_end) {
    const uint32_t z = (uint32_t)(c.valid - 1 - prev) + carry;
    if (z) emit_run(z, s);
  }
}

// ---- K-hist ----------------------------------------------------------------------------------
struct HistSink {
  uint32_t *h;
  __device__ __forceinline__ void tok(int sym, uint32_t, int) { atomicAdd(&h[sym], 1u); }
};

// grid (nseg, n).  seghist: [n][nseg][261].
__global__ void __launch_bounds__(kHuffThreads)
    k_huff_hist(const uint8_t *__restrict__ in, HuffGeom hg, uint32_t *__restrict__ seghist) {
  __shared__ uint32_t sh[kSyms];
  __shared__ uint32_t ws[17];
  __shared__ uint32_t rows[kHuffThreads * kRowWords];
  for (int i = threadIdx.x; i < kSyms; i += blockDim.x) sh[i] = 0;
  __syncthreads();
  const uint8_t *seg = in + (size_t)blockIdx.y * hg.in_stride + (size_t)blockIdx.x * hg.seg_size;
  uint32_t carry = 0;
  HistSink sink{sh};
  for (int base = 0; base < hg.seg_size; base += kPieceBytes) {
    const int off = base + threadIdx.x * kChunkBytes;
    Chunk c;
    load_chunk(c, rows, seg, hg.seg_size, off);
    uint32_t carry_out;
    const uint32_t z_in = block_run_scan(run_summary(c), carry, ws, &carry_out);
    carry = carry_out;
    walk_chunk(c, z_in, c.valid > 0 && off + c.valid == hg.seg_size, sink);
  }
  __syncthreads();
  uint32_t *dst = seghist + ((size_t)blockIdx.y * hg.nseg + blockIdx.x) * kSyms;
  for (int i = threadIdx.x; i < kSyms; i += blockDim.x) dst[i] = sh[i];
}

// =================================================================================================
// Balanced tokenisation (v2).  The walks above cost as much as the densest lane of a warp, and the
// coefficient planes are very uneven (dense low frequencies, empty high frequencies).  Here the
// non-zero bytes of a piece ("items") are first compacted into a position list in shared memory;
// warps then take equal numbers of items.  Item k stands for [zero-run of gap_k bytes][literal]:
// gap_0 = p_0 + zeros carried in, gap_k = p_k - p_(k-1) - 1.  The run that is still open at the end
// of a piece is carried to the next piece; at the segment end it is emitted by one thread.
// =================================================================================================
#ifndef HIMG_TOK_THREADS
#define HIMG_TOK_THREADS 256
#endif
constexpr int kTokThreads = HIMG_TOK_THREADS;
constexpr int kTokPiece = kTokThreads * kChunkBytes;  // 8 KiB
constexpr int kTokWarps = kTokThreads / 32;

struct PieceItems {
  int count;        // number of items (non-zero bytes) in the piece
  int len;          // valid bytes in the piece
  uint32_t zeros_in;  // zeros carried in from earlier pieces
};

// Loads one piece, builds rows (for byte lookups) and the item position list.  Returns the zeros
// carried out.  `ipos` holds kTokPiece u16, `ws` 9 words.  Ends with a barrier.
__device__ __forceinline__ uint32_t build_items(const uint8_t *__restrict__ seg, int seg_size, int base, uint32_t *rows,
                                                unsigned short *ipos, uint32_t *ws, uint32_t zeros_in, PieceItems *P) {
  Chunk c;
  load_chunk(c, rows, seg, seg_size, base + (int)threadIdx.x * kChunkBytes);
  uint32_t total;
  const uint32_t first = block_exscan_u32((uint32_t)__popc(c.nz), ws, &total);
  uint32_t m = c.nz, k = first;
  const int pbase = (int)threadIdx.x * kChunkBytes;
  while (m) {
    ipos[k++] = (unsigned short)(pbase + __ffs(m) - 1);
    m &= m - 1;
  }
  __syncthreads();
  P->count = (int)total;
  P->len = min(kTokPiece, seg_size - base);
  P->zeros_in = zeros_in;
  return total ? (uint32_t)(P->len - 1 - (int)ipos[total - 1]) : zeros_in + (uint32_t)P->len;
}

__device__ __forceinline__ uint32_t item_byte(const uint32_t *rows, int pos) {
  return reinterpret_cast<const uint8_t *>(rows)[(pos >> 5) * (kRowWords * 4) + (pos & 31)];
}
__device__ __forceinline__ uint32_t item_gap(const unsigned short *ipos, int k, uint32_t zeros_in) {
  return k ? (uint32_t)(ipos[k] - ipos[k - 1] - 1) : (uint32_t)ipos[0] + zeros_in;
}

// run length -> (symbol, extra bits value) of the LAST token of the run (after full 16662 tokens)
__device__ __forceinline__ int run_symbol(uint32_t z, uint32_t *extra) {
  if (z == 1) { *extra = 0; return 0; }
  if (z == 2) { *extra = 0; return 256; }
  if (z <= 6) { *extra = z - 3; return 257; }
  if (z <= 22) { *extra = z - 7; return 258; }
  if (z <= 278) { *extra = z - 23; return 259; }
  *extra = z - 279;
  return 260;
}

// Number of zero bytes immediately before byte `pos` of a segment (block-cooperative, uniform
// result): the run that is open where a part starts.  Usually one 2 KiB look-back.
__device__ __forceinline__ uint32_t zeros_before(const uint8_t *__restrict__ seg, int pos, int *s_last) {
  uint32_t zeros = 0;
  int end = pos;
  while (end > 0) {
    const int win = min(end, kTokThreads * 8), start = end - win;
    if (threadIdx.x == 0) *s_last = -1;
    __syncthreads();
    int last = -1;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int i = start + 8 * (int)threadIdx.x + k;
      if (i < end && seg[i]) last = i;
    }
    if (last >= 0) atomicMax(s_last, last);
    __syncthreads();
    const int l = *s_last;
    __syncthreads();
    if (l >= 0) return zeros + (uint32_t)(end - 1 - l);
    zeros += (uint32_t)win;
    end = start;
  }
  return zeros;
}

// ORs a byte into global memory (bytes shared by two parts of a segment; pre-zeroed by k_huff_layout)
__device__ __forceinline__ void atomic_or_byte(uint8_t *p, uint32_t v) {
  const uintptr_t a = reinterpret_cast<uintptr_t>(p);
  atomicOr(reinterpret_cast<uint32_t *>(a & ~(uintptr_t)3), (v & 0xffu) << (8 * (a & 3)));
}

// Item lists handed from the histogram pass to the packer.  Both kernels cut a part into the same 8 KiB
// pieces and need the same list of non-zero bytes per piece; building it (load, non-zero masks, block
// scan, compaction) was 40 % of the packer's time.  k_huff_hist2 therefore stores the list of every
// piece that holds at most kItemCap items (position inside the piece + byte value: 3 bytes per item,
// ~0.4 bytes per coefficient byte at quality 50) and the packer reads it back instead of the planes.
// Denser pieces are marked and rebuilt from the planes as before.
constexpr int kItemCap = 2048;
constexpr uint32_t kItemsNotStored = 0xffffffffu;
struct ItemLists {
  unsigned short *pos;  // [slots][kItemCap]
  uint8_t *val;         // [slots][kItemCap]
  uint32_t *count;      // [slots]; kItemsNotStored: rebuild from the planes
  int pieces_per_part;  // slots of one (item, segment, part); 0: no lists (every piece is rebuilt)
};
__device__ __forceinline__ size_t item_slot(const ItemLists &L, const HuffGeom &hg, int item, int piece) {
  return ((size_t)item * hg.nseg * hg.nsub + blockIdx.x) * L.pieces_per_part + piece;
}

// grid (nseg * nsub, n), block kTokThreads.  seghist: [n][nseg * nsub][261].  MIXED: see MixedHuff.
template <bool MIXED = false>
__global__ void __launch_bounds__(kTokThreads, 8)
    k_huff_hist2(const uint8_t *__restrict__ in, HuffGeom hg, uint32_t *__restrict__ seghist, ItemLists lists,
                 uint32_t *__restrict__ total, MixedHuff mh = {}) {
  __shared__ uint32_t sh[kSyms];
  __shared__ uint32_t ws[kTokWarps + 1];
  __shared__ uint32_t rows[kTokThreads * kRowWords];
  __shared__ unsigned short ipos[kTokPiece];
  __shared__ int s_last;
  for (int i = threadIdx.x; i < kSyms; i += blockDim.x) sh[i] = 0;
  __syncthreads();
  const int b = blockIdx.x / hg.nsub, part = blockIdx.x - b * hg.nsub;
  HuffGeom ig = hg;  // this item's chunk
  const bool idle = MIXED && !(mixed_chunk(mh, blockIdx.y, ig) && b < ig.nseg);  // (a zero histogram row)
  const uint8_t *seg0 = in + (size_t)blockIdx.y * hg.in_stride + (size_t)b * ig.seg_size;
  const int p0 = part * ig.sub_size, plen = idle ? 0 : min(ig.sub_size, ig.seg_size - p0);
  const uint8_t *seg = seg0 + p0;
  uint32_t carry = part ? zeros_before(seg0, p0, &s_last) : 0u;
  for (int base = 0; base < plen; base += kTokPiece) {
    PieceItems P;
    carry = build_items(seg, plen, base, rows, ipos, ws, carry, &P);
    const bool keep = lists.pieces_per_part != 0 && P.count <= kItemCap;
    const size_t slot = lists.pieces_per_part ? item_slot(lists, hg, blockIdx.y, base / kTokPiece) : 0;
    if (lists.pieces_per_part && threadIdx.x == 0) lists.count[slot] = keep ? (uint32_t)P.count : kItemsNotStored;
    for (int k = threadIdx.x; k < P.count; k += kTokThreads) {
      uint32_t z = item_gap(ipos, k, P.zeros_in), ex;
      while (z >= (uint32_t)kMaxRun) {
        atomicAdd(&sh[260], 1u);
        z -= kMaxRun;
      }
      if (z) atomicAdd(&sh[run_symbol(z, &ex)], 1u);
      const uint32_t v = item_byte(rows, ipos[k]);
      atomicAdd(&sh[v], 1u);
      if (keep) {
        lists.pos[slot * kItemCap + k] = ipos[k];
        lists.val[slot * kItemCap + k] = (uint8_t)v;
      }
    }
    __syncthreads();  // rows / ipos are rewritten by the next piece
  }
  if (threadIdx.x == 0 && carry && part == hg.nsub - 1) {  // the run still open at the segment end
    uint32_t z = carry, ex;
    while (z >= (uint32_t)kMaxRun) {
      atomicAdd(&sh[260], 1u);
      z -= kMaxRun;
    }
    if (z) atomicAdd(&sh[run_symbol(z, &ex)], 1u);
  }
  __syncthreads();
  uint32_t *dst = seghist + ((size_t)blockIdx.y * hg.nseg * hg.nsub + blockIdx.x) * kSyms;
  for (int i = threadIdx.x; i < kSyms; i += blockDim.x) {
    const uint32_t v = sh[i];
    dst[i] = v;
    // the chunk's histogram (what the tree is built from): summed here, so that k_huff_tree does not
    // walk over the rows -- a chain of dependent L2 round trips, the longest part of it for tall images
    if (total && v) atomicAdd(&total[(size_t)blockIdx.y * kSyms + i], v);
  }
}

// ---- K-tree ----------------------------------------------------------------------------------
constexpr int kTreeThreads = 288;

// The (up to two) chunks of an image get their trees in ONE launch: the construction is a serial
// chain of ~80 us per tree, and two CTAs run it side by side.
struct TreeParams {
  const uint32_t *total[2];    // [n][261] chunk histograms summed by k_huff_hist2, or null: sum the rows here
  const uint32_t *seghist[2];  // [n][rows][261]
  TreeOut *trees[2];           // [n]
  int rows[2];                 // histogram rows per item (segments x parts)
};

// grid (n, chunks).  err: set to HIMGCU_ERR_UNSUPPORTED (5) if a code exceeds 32 bits.
//
// The construction is a serial chain (n - 1 merges), so what counts is the latency of ONE thread's loop:
//  * merge: the heads of both queues live in registers (count and node of the next leaf, count and range of
//    the front group of internal nodes); a pick costs one shared-memory load, a new node three stores;
//  * codes, depths and the positions of the serialised tree need no stack and no second serial pass: the
//    merge records parent links and subtree sizes in bits (leaf = 10, branch = 1 + both), and every LEAF
//    then walks up its parent chain in parallel: the branch bits arrive deepest first (shifted in from the
//    right they are the code), the pre-order position is 1 per ancestor + the left sibling subtree wherever
//    the path turns right; it writes its code table entry and its 10 bits of the tree.
// (Round 1 walked a stack in shared memory: 65 us for the merge + 35 us for the serialisation of a
// 261-leaf tree.)
__global__ void __launch_bounds__(kTreeThreads)
    k_huff_tree(const TreeParams P, int *err) {
  __shared__ uint32_t cnt[kMaxNodes];
  __shared__ uint32_t kids[kMaxNodes];  // internal node: child a | child b << 16
  __shared__ short nsym[kSyms];         // leaf node -> symbol
  __shared__ short lq[kSyms + 1];       // leaves in (count ascending, index DEscending) order
  __shared__ uint32_t lcnt[kSyms + 1];  // their counts
  __shared__ short ist[kSyms], gend[kSyms];
  __shared__ unsigned short bsize[kMaxNodes];  // serialised size of the subtree in bits
  __shared__ short par[kMaxNodes];             // 2 * parent + (second child ? 1 : 0); -1 for the root
  __shared__ uint32_t s_code[kSyms];
  __shared__ uint8_t s_len[kSyms + 3];
  __shared__ uint32_t s_tree[kTreeBytesMax / 4];
  __shared__ uint32_t warp_tot[kTreeThreads / 32 + 1];
  __shared__ int s_nleaves, s_bits;

  const int t = threadIdx.x;
  const uint32_t *__restrict__ seghist = P.seghist[blockIdx.y];
  const int nseg = P.rows[blockIdx.y];
  TreeOut *out = P.trees[blockIdx.y] + blockIdx.x;
  // 1. chunk histogram = sum of its segments' histograms (coalesced across threads)
  uint32_t my = 0;
  if (t < kSyms) {
    if (P.total[blockIdx.y]) {
      my = P.total[blockIdx.y][(size_t)blockIdx.x * kSyms + t];
    } else {
      // independent loads, eight in flight
      const uint32_t *p = seghist + (size_t)blockIdx.x * nseg * kSyms + t;
      int s = 0;
      for (; s + 8 <= nseg; s += 8) {
        uint32_t v[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) v[k] = __ldg(p + (size_t)(s + k) * kSyms);
#pragma unroll
        for (int k = 0; k < 8; ++k) my += v[k];
      }
      for (; s < nseg; ++s) my += __ldg(p + (size_t)s * kSyms);
    }
    out->hist[t] = my;
    s_code[t] = 0;
    s_len[t] = 0;
  }
  for (int i = t; i < kTreeBytesMax / 4; i += blockDim.x) s_tree[i] = 0;
  // 2. leaves = used symbols in symbol order (huffman_enc.cpp:186-196)
  uint32_t total;
  const uint32_t li = block_exscan_u32(t < kSyms && my ? 1u : 0u, warp_tot, &total);
  if (t < kSyms && my) {
    cnt[li] = my;
    nsym[li] = (short)t;
    bsize[li] = 10;  // bit 1 + the 9-bit symbol
  }
  if (t == 0) s_nleaves = (int)total;
  __syncthreads();
  const int n = s_nleaves;
  // 3. rank sort under (count ascending, index DEscending): keys are unique
  if (t < n) {
    const uint32_t c = cnt[t];
    int rank = 0;
    for (int j = 0; j < n; ++j) {
      const uint32_t cj = cnt[j];
      rank += (cj < c || (cj == c && j > t)) ? 1 : 0;
    }
    lq[rank] = (short)t;
    lcnt[rank] = c;
  }
  if (t == 0) lq[n] = 0, lcnt[n] = 0;  // (read ahead by the merge, never used)
  __syncthreads();
  if (t == 0 && n > 0) {
    // 4. two-queue merge.  The reference picks the minimum under (count ascending, node index DEscending)
    //    (huffman_enc.cpp:199-227).  Internal nodes are created with non-decreasing counts, so they form
    //    groups of equal count in creation order: the FRONT group is consumed first, newest node first,
    //    and an internal node beats a leaf of equal count.  While the front group is also the LAST one it
    //    is a stack that new nodes of the same count are still pushed onto.
    int root = lq[0];
    if (n > 1) {
      int ist_n = 0, lp = 0, next = n;
      int fstart = 0, ftop = 0, fend = 0;  // front group [fstart, ftop) of ist, closed end fend (unless it is the last group)
      uint32_t fcount = 0;
      bool front_is_last = true;
      int last_start = 0;
      uint32_t last_count = 0;
      uint32_t lc = lcnt[0];
      int lnode = lq[0];
      for (int merge = 0; merge < n - 1; ++merge) {
        int pick[2];
        uint32_t pc[2];
#pragma unroll
        for (int k = 0; k < 2; ++k) {
          int top = front_is_last ? ist_n : ftop;
          const bool take_int = top > fstart && (lp >= n || fcount <= lc);
          if (take_int) {
            --top;
            pick[k] = ist[top];
            pc[k] = fcount;
            if (front_is_last) {
              ist_n = top;
            } else {
              ftop = top;
              if (ftop == fstart) {  // exhausted: the next group in creation order
                fstart = fend;
                if (fstart == last_start) {
                  front_is_last = true;
                  fcount = last_count;
                } else {
                  ftop = fend = gend[fstart];
                  fcount = cnt[ist[fstart]];
                }
              }
            }
          } else {
            pick[k] = lnode;
            pc[k] = lc;
            ++lp;
            lc = lcnt[lp];
            lnode = lq[lp];
          }
        }
        root = next++;
        const uint32_t c = pc[0] + pc[1];
        kids[root] = (uint32_t)pick[0] | ((uint32_t)pick[1] << 16);
        cnt[root] = c;
        par[pick[0]] = (short)(2 * root);
        par[pick[1]] = (short)(2 * root + 1);
        bsize[root] = (unsigned short)(1u + bsize[pick[0]] + bsize[pick[1]]);
        if (ist_n > last_start && last_count == c) {
          ist[ist_n++] = (short)root;
        } else if (ist_n == last_start) {  // the last group is empty: it restarts with this count
          last_count = c;
          if (front_is_last) fcount = c;
          ist[ist_n++] = (short)root;
        } else {  // close the last group, open a new one
          gend[last_start] = (short)ist_n;
          if (front_is_last) {
            front_is_last = false;
            ftop = fend = ist_n;
          }
          last_start = ist_n;
          last_count = c;
          ist[ist_n++] = (short)root;
        }
      }
    }
    par[root] = -1;
    s_bits = bsize[root];
  }
  if (t == 0 && n == 0) s_bits = 0;
  __syncthreads();
  // 5. every leaf: depth, code and pre-order position by a walk up its parent chain (huffman_enc.cpp:148-180,
  //    :229-237: bit 0, first subtree, second subtree; the second child's code has bit `depth of the parent`
  //    set), then its entry of the code table and its 10 bits of the serialised tree.  A single leaf gets a
  //    1-bit code.
  if (t < n) {
    int bits = 0, cur = t;
    uint32_t cd = 0, p = 0;
    for (int sl = par[cur]; sl >= 0; sl = par[cur]) {
      const int up = sl >> 1;
      cd = (cd << 1) | (uint32_t)(sl & 1);  // (bits beyond 32 fall off: such a tree is refused below)
      p += 1u + ((sl & 1) ? (uint32_t)bsize[kids[up] & 0xffffu] : 0u);
      cur = up;
      ++bits;
    }
    if (n == 1) bits = 1;
    const int sym = nsym[t];
    s_code[sym] = cd;
    s_len[sym] = (uint8_t)min(bits, 255);
    if (bits > 32) atomicMax(err, 5);
    const uint32_t v = 1u | ((uint32_t)sym << 1), sh = p & 31;
    atomicOr(&s_tree[p >> 5], v << sh);
    if (sh > 22) atomicOr(&s_tree[(p >> 5) + 1], v >> (32 - sh));
  }
  __syncthreads();
  if (t < kSyms) {
    out->code[t] = s_code[t];
    out->len[t] = s_len[t];
  }
  for (int i = t; i < kTreeBytesMax; i += blockDim.x) out->tree[i] = (uint8_t)(s_tree[i >> 2] >> (8 * (i & 3)));
  if (t == 0) {
    out->tree_bits = (uint32_t)s_bits;
    out->nleaves = (uint32_t)n;
  }
}

// ---- K-layout --------------------------------------------------------------------------------
struct LayoutChunk {
  const uint32_t *part_bits;  // [n][nseg][nsub] bits of every part (k_huff_segbits)
  const uint32_t *seghist;  // [n][nseg][261]
  const TreeOut *trees;     // [n]
  uint32_t *seg_bits;       // [n][nseg] out
  uint32_t *seg_pos;        // [n][nseg] out: absolute offset of the segment PAYLOAD inside the item
  uint32_t *part_start;     // [n][nseg][nsub] out: first bit of every part inside its segment
  int nsub;
  const uint8_t *prefix;    // bytes emitted before the chunk (container headers), may be null
  int prefix_len;
  int size_patch;           // offset inside the prefix of the u32 chunk size, or -1
  int nseg;
  int framed;               // segments carry 2/4-byte size headers (huffman_enc.cpp:340-352)
};
struct LayoutParams {
  LayoutChunk ch[2];
  int nchunks;
  int riff_patch;  // patch u32 at item offset 4 with (total - 8)
  uint8_t *out;
  unsigned long long out_stride;
  uint32_t *sizes;  // [n]; 0 = does not fit
  int *err;
};

constexpr int kLayoutThreads = 256;

// Bits of every part of every segment = its histogram . (code length + extra bits): a warp per histogram row.
// (One CTA per image used to do this inside k_huff_layout: 100 us for the 1024 rows of a single 8K image.)
// grid (ceil(rows / 8), n), block 256.
__global__ void __launch_bounds__(256) k_huff_segbits(const uint32_t *__restrict__ seghist, const TreeOut *__restrict__ trees,
                                                      int rows, uint32_t *__restrict__ part_bits) {
  const int item = blockIdx.y, lane = threadIdx.x & 31, row = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= rows) return;
  const TreeOut *tr = trees + item;
  const uint32_t *h = seghist + ((size_t)item * rows + row) * kSyms;
  unsigned long long pb = 0;
#pragma unroll
  for (int k = 0; k < (kSyms + 31) / 32; ++k) {
    const int s = lane + 32 * k;
    if (s < kSyms) pb += (unsigned long long)__ldg(h + s) * (uint32_t)(tr->len[s] + sym_extra_bits(s));
  }
#pragma unroll
  for (int d = 16; d >= 1; d >>= 1) pb += __shfl_xor_sync(0xffffffffu, pb, d);
  if (lane == 0) part_bits[(size_t)item * rows + row] = (uint32_t)pb;
}

__device__ __forceinline__ void put_u32le(uint8_t *p, uint32_t x) {
  p[0] = (uint8_t)x;
  p[1] = (uint8_t)(x >> 8);
  p[2] = (uint8_t)(x >> 16);
  p[3] = (uint8_t)(x >> 24);
}

// grid (n).
__global__ void __launch_bounds__(kLayoutThreads) k_huff_layout(const __grid_constant__ LayoutParams P) {
  __shared__ uint32_t ws[kLayoutThreads / 32 + 1];
  __shared__ unsigned long long s_chunk_bytes[2];
  __shared__ int s_too_long;
  const int item = blockIdx.x, t = threadIdx.x, lane = t & 31;
  uint8_t *out = P.out + (size_t)item * P.out_stride;
  if (t == 0) s_too_long = 0;

  // pass 1: segment bit lengths and chunk sizes
  for (int k = 0; k < P.nchunks; ++k) {
    const LayoutChunk &C = P.ch[k];
    const TreeOut *tr = C.trees + item;
    __syncthreads();
    for (int s = t; s < kSyms; s += blockDim.x)
      if (tr->len[s] > 32) s_too_long = 1;  // the reference's codes are uint32_t (huffman_enc.cpp:179): unsupported
    if (t == 0) s_chunk_bytes[k] = 0;
    __syncthreads();
    unsigned long long mine = 0;
    for (int b = t; b < C.nseg; b += kLayoutThreads) {  // a thread per segment: running sum over its parts
      unsigned long long bits = 0;
      for (int part = 0; part < C.nsub; ++part) {
        const size_t pi = ((size_t)item * C.nseg + b) * C.nsub + part;
        C.part_start[pi] = (uint32_t)bits;
        bits += C.part_bits[pi];
      }
      C.seg_bits[(size_t)item * C.nseg + b] = (uint32_t)bits;
      const unsigned long long sz = (bits + 7) >> 3;
      mine += sz + (C.framed ? (sz <= 0x7fff ? 2 : 4) : 0);
    }
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, d);
    if (lane == 0 && mine) atomicAdd(&s_chunk_bytes[k], mine);
  }
  __syncthreads();
  unsigned long long total = 0;
  for (int k = 0; k < P.nchunks; ++k)
    total += (unsigned long long)P.ch[k].prefix_len + ((P.ch[k].trees[item].tree_bits + 7) >> 3) + s_chunk_bytes[k];
  if (s_too_long || total > P.out_stride || total > 0xffffffffull) {
    // size 0 marks the item as not encoded (the packer skips it, the host calls report it); the flag
    // says why: 5 = a Huffman code longer than 32 bits, 4 = the output does not fit
    if (t == 0) {
      P.sizes[item] = 0;
      atomicMax(P.err, s_too_long ? 5 : 4);
    }
    return;
  }

  // pass 2: emit prefixes, trees, segment headers; record payload positions
  uint32_t pos = 0;
  for (int k = 0; k < P.nchunks; ++k) {
    const LayoutChunk &C = P.ch[k];
    const TreeOut *tr = C.trees + item;
    const uint32_t prefix_at = pos;
    for (int i = t; i < C.prefix_len; i += blockDim.x) out[pos + i] = C.prefix[i];
    pos += C.prefix_len;
    const uint32_t tree_bytes = (tr->tree_bits + 7) >> 3;
    for (int i = t; i < (int)tree_bytes; i += blockDim.x) out[pos + i] = tr->tree[i];
    const uint32_t chunk_bytes = tree_bytes + (uint32_t)s_chunk_bytes[k];
    __syncthreads();  // prefix bytes written before the patch below
    if (t == 0 && C.size_patch >= 0) put_u32le(out + prefix_at + C.size_patch, chunk_bytes);
    pos += tree_bytes;
    // exclusive scan of (header + payload) over the segments, kLayoutThreads at a time
    uint32_t run = 0;
    for (int b0 = 0; b0 < C.nseg; b0 += kLayoutThreads) {
      const int b = b0 + t;
      uint32_t sz = 0, hdr = 0;
      if (b < C.nseg) {
        sz = (C.seg_bits[(size_t)item * C.nseg + b] + 7) >> 3;
        hdr = C.framed ? (sz <= 0x7fff ? 2u : 4u) : 0u;
      }
      uint32_t tot;
      const uint32_t ex = block_exscan_u32(sz + hdr, ws, &tot);
      if (b < C.nseg) {
        uint8_t *h = out + pos + run + ex;
        if (hdr == 2) {
          h[0] = (uint8_t)sz;
          h[1] = (uint8_t)(sz >> 8);
        } else if (hdr == 4) {
          const uint32_t lo = (sz & 0x7fff) | 0x8000, hi = sz >> 15;
          h[0] = (uint8_t)lo;
          h[1] = (uint8_t)(lo >> 8);
          h[2] = (uint8_t)hi;
          h[3] = (uint8_t)(hi >> 8);
        }
        C.seg_pos[(size_t)item * C.nseg + b] = pos + run + ex + hdr;
        // a byte shared by two parts is written with atomicOr from both sides: clear it
        for (int part = 1; part < C.nsub; ++part) {
          const uint32_t st = C.part_start[((size_t)item * C.nseg + b) * C.nsub + part];
          if (st & 7) out[pos + run + ex + hdr + (st >> 3)] = 0;
        }
      }
      run += tot;
    }
    pos += run;
  }
  if (t == 0) {
    P.sizes[item] = pos;
    if (P.riff_patch) put_u32le(out + 4, pos - 8);
  }
}

// Device error flag value of an image whose dims are out of bounds (a mixed batch): below the others (4, 5, 99), so
// that under atomicMax a worse error of the same call still wins.
constexpr int kEncErrDims = 1;

// k_huff_layout of a mixed-geometry batch, grid (n).  Chunk 0 is the LRES chunk, chunk 1 the FRES chunk; C.nseg is the bounding segment
// count, the slot stride of the segment tables; item i's chunks have their own segment counts (1, gi.rows) and the
// FRES chunk is framed only when gi.rows > 1.  Its width and height go into the two u32 at offset frmt_at of chunk 0's
// prefix.  An image whose dims are out of bounds gets size 0 and the flag kEncErrDims.  (A kernel of its own: the
// smallest change to k_huff_layout's source moves its register allocation.)
__global__ void __launch_bounds__(kLayoutThreads)
    k_huff_layout_mixed(const __grid_constant__ LayoutParams P, MixedDims md, int frmt_at) {
  __shared__ uint32_t ws[kLayoutThreads / 32 + 1];
  __shared__ unsigned long long s_chunk_bytes[2];
  __shared__ int s_too_long;
  const int item = blockIdx.x, t = threadIdx.x, lane = t & 31;
  uint8_t *out = P.out + (size_t)item * P.out_stride;
  if (t == 0) s_too_long = 0;
  Geom gi;
  if (!image_geom(md, item, gi)) {
    if (t == 0) {
      P.sizes[item] = 0;
      atomicMax(P.err, kEncErrDims);
    }
    return;
  }

  // pass 1: segment bit lengths and chunk sizes
  for (int k = 0; k < P.nchunks; ++k) {
    const LayoutChunk &C = P.ch[k];
    const TreeOut *tr = C.trees + item;
    __syncthreads();
    for (int s = t; s < kSyms; s += blockDim.x)
      if (tr->len[s] > 32) s_too_long = 1;  // the reference's codes are uint32_t (huffman_enc.cpp:179): unsupported
    if (t == 0) s_chunk_bytes[k] = 0;
    __syncthreads();
    unsigned long long mine = 0;
    const int nseg = k ? gi.rows : 1, framed = k && gi.rows > 1;  // this item's chunk
    for (int b = t; b < nseg; b += kLayoutThreads) {  // a thread per segment: running sum over its parts
      unsigned long long bits = 0;
      for (int part = 0; part < C.nsub; ++part) {
        const size_t pi = ((size_t)item * C.nseg + b) * C.nsub + part;
        C.part_start[pi] = (uint32_t)bits;
        bits += C.part_bits[pi];
      }
      C.seg_bits[(size_t)item * C.nseg + b] = (uint32_t)bits;
      const unsigned long long sz = (bits + 7) >> 3;
      mine += sz + (framed ? (sz <= 0x7fff ? 2 : 4) : 0);
    }
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, d);
    if (lane == 0 && mine) atomicAdd(&s_chunk_bytes[k], mine);
  }
  __syncthreads();
  unsigned long long total = 0;
  for (int k = 0; k < P.nchunks; ++k)
    total += (unsigned long long)P.ch[k].prefix_len + ((P.ch[k].trees[item].tree_bits + 7) >> 3) + s_chunk_bytes[k];
  if (s_too_long || total > P.out_stride || total > 0xffffffffull) {
    // size 0 marks the item as not encoded (the packer skips it, the host calls report it); the flag
    // says why: 5 = a Huffman code longer than 32 bits, 4 = the output does not fit
    if (t == 0) {
      P.sizes[item] = 0;
      atomicMax(P.err, s_too_long ? 5 : 4);
    }
    return;
  }

  // pass 2: emit prefixes, trees, segment headers; record payload positions
  uint32_t pos = 0;
  for (int k = 0; k < P.nchunks; ++k) {
    const LayoutChunk &C = P.ch[k];
    const TreeOut *tr = C.trees + item;
    const uint32_t prefix_at = pos;
    for (int i = t; i < C.prefix_len; i += blockDim.x) out[pos + i] = C.prefix[i];
    pos += C.prefix_len;
    const uint32_t tree_bytes = (tr->tree_bits + 7) >> 3;
    for (int i = t; i < (int)tree_bytes; i += blockDim.x) out[pos + i] = tr->tree[i];
    const uint32_t chunk_bytes = tree_bytes + (uint32_t)s_chunk_bytes[k];
    __syncthreads();  // prefix bytes written before the patch below
    if (t == 0 && C.size_patch >= 0) put_u32le(out + prefix_at + C.size_patch, chunk_bytes);
    if (t == 0 && k == 0) {
      put_u32le(out + prefix_at + frmt_at, (uint32_t)gi.w);
      put_u32le(out + prefix_at + frmt_at + 4, (uint32_t)gi.h);
    }
    pos += tree_bytes;
    // exclusive scan of (header + payload) over the segments, kLayoutThreads at a time
    uint32_t run = 0;
    const int nseg = k ? gi.rows : 1, framed = k && gi.rows > 1;  // this item's chunk
    for (int b0 = 0; b0 < nseg; b0 += kLayoutThreads) {
      const int b = b0 + t;
      uint32_t sz = 0, hdr = 0;
      if (b < nseg) {
        sz = (C.seg_bits[(size_t)item * C.nseg + b] + 7) >> 3;
        hdr = framed ? (sz <= 0x7fff ? 2u : 4u) : 0u;
      }
      uint32_t tot;
      const uint32_t ex = block_exscan_u32(sz + hdr, ws, &tot);
      if (b < nseg) {
        uint8_t *h = out + pos + run + ex;
        if (hdr == 2) {
          h[0] = (uint8_t)sz;
          h[1] = (uint8_t)(sz >> 8);
        } else if (hdr == 4) {
          const uint32_t lo = (sz & 0x7fff) | 0x8000, hi = sz >> 15;
          h[0] = (uint8_t)lo;
          h[1] = (uint8_t)(lo >> 8);
          h[2] = (uint8_t)hi;
          h[3] = (uint8_t)(hi >> 8);
        }
        C.seg_pos[(size_t)item * C.nseg + b] = pos + run + ex + hdr;
        // a byte shared by two parts is written with atomicOr from both sides: clear it
        for (int part = 1; part < C.nsub; ++part) {
          const uint32_t st = C.part_start[((size_t)item * C.nseg + b) * C.nsub + part];
          if (st & 7) out[pos + run + ex + hdr + (st >> 3)] = 0;
        }
      }
      run += tot;
    }
    pos += run;
  }
  if (t == 0) {
    P.sizes[item] = pos;
    if (P.riff_patch) put_u32le(out + 4, pos - 8);
  }
}

// ---- K-pack ----------------------------------------------------------------------------------
struct SizeSink {
  const uint32_t *lenx;  // len + extra bits per symbol
  uint32_t bits;
  __device__ __forceinline__ void tok(int sym, uint32_t, int) { bits += lenx[sym]; }
};

// Thread-local LSB-first bit accumulator writing into a shared-memory window.  Only tokens whose
// first bit falls inside [w0, w0 + kWinBits) are written (a token may spill <= 46 bits into the
// two slack words).
struct EmitSink {
  const uint32_t *code;
  const uint8_t *len;
  uint32_t *win;
  uint32_t pos;  // position of the next token, in window coordinates of the whole piece
  uint32_t w0;
  uint64_t acc;
  int nacc;   // bits held in acc; -1 = accumulator not positioned yet
  int wpos;
  __device__ __forceinline__ void put(uint32_t v, int n) {
    acc |= (uint64_t)v << nacc;
    nacc += n;
    if (nacc >= 32) {
      atomicOr(&win[wpos++], (uint32_t)acc);
      acc >>= 32;
      nacc -= 32;
    }
  }
  __device__ __forceinline__ void tok(int sym, uint32_t extra, int nextra) {
    const int l = len[sym];
    if (pos >= w0 && pos < w0 + (uint32_t)kWinBits) {
      if (nacc < 0) {
        const uint32_t rel = pos - w0;
        nacc = (int)(rel & 31);
        wpos = (int)(rel >> 5);
        acc = 0;
      }
      if (l) put(code[sym], l);
      if (nextra) put(extra, nextra);
    } else if (nacc >= 0) {
      flush();
    }
    pos += (uint32_t)(l + nextra);
  }
  __device__ __forceinline__ void flush() {
    if (nacc > 0) atomicOr(&win[wpos], (uint32_t)acc);
    nacc = -1;
  }
};

// grid (nseg, n).  Dynamic shared memory: (kWinWords + 2) words.
__global__ void __launch_bounds__(kHuffThreads)
    k_huff_pack(const uint8_t *__restrict__ in, HuffGeom hg, const TreeOut *__restrict__ trees,
                const uint32_t *__restrict__ seg_bits, const uint32_t *__restrict__ seg_pos,
                const uint32_t *__restrict__ sizes, uint8_t *__restrict__ out,
                unsigned long long out_stride, int *err) {
  extern __shared__ uint32_t win[];
  __shared__ uint32_t s_code[kSyms];
  __shared__ uint8_t s_len[kSyms + 3];
  __shared__ uint32_t s_lenx[kSyms];
  __shared__ uint32_t ws[17];
  __shared__ uint32_t rows[kHuffThreads * kRowWords];
  const int item = blockIdx.y, b = blockIdx.x, t = threadIdx.x;
  if (sizes[item] == 0) return;  // did not fit (k_huff_layout)
  const TreeOut *tr = trees + item;
  for (int s = t; s < kSyms; s += blockDim.x) {
    s_code[s] = tr->code[s];
    s_len[s] = tr->len[s];
    s_lenx[s] = (uint32_t)tr->len[s] + sym_extra_bits(s);
  }
  for (int i = t; i < kWinWords + 2; i += blockDim.x) win[i] = 0;
  __syncthreads();
  const uint8_t *seg = in + (size_t)item * hg.in_stride + (size_t)b * hg.seg_size;
  uint8_t *dst = out + (size_t)item * out_stride + seg_pos[(size_t)item * hg.nseg + b];

  uint32_t carry = 0;       // zeros of an unfinished run
  uint32_t gbits = 0;       // bits emitted so far (complete bytes below gbits>>3 are in `dst`)
  for (int base = 0; base < hg.seg_size; base += kPieceBytes) {
    const int off = base + t * kChunkBytes;
    Chunk c;
    load_chunk(c, rows, seg, hg.seg_size, off);
    uint32_t carry_out;
    const uint32_t z_in = block_run_scan(run_summary(c), carry, ws, &carry_out);
    carry = carry_out;
    const bool last = c.valid > 0 && off + c.valid == hg.seg_size;
    SizeSink ss{s_lenx, 0};
    walk_chunk(c, z_in, last, ss);
    uint32_t piece_bits;
    const uint32_t my_start = block_exscan_u32(ss.bits, ws, &piece_bits);
    // window coordinates: bit 0 of the window = byte boundary at or below gbits
    const uint32_t lead = gbits & 7;
    const uint32_t vend = lead + piece_bits;
    const uint32_t gbyte = gbits >> 3;
    for (uint32_t w0 = 0; w0 < vend || w0 == 0; w0 += kWinBits) {
      if (ss.bits && lead + my_start < w0 + (uint32_t)kWinBits && lead + my_start + ss.bits > w0) {
        EmitSink es{s_code, s_len, win, lead + my_start, w0, 0, -1, 0};
        walk_chunk(c, z_in, last, es);
        es.flush();
      }
      __syncthreads();
      const bool last_win = w0 + (uint32_t)kWinBits >= vend;
      const uint32_t nbytes = last_win ? ((vend - w0) >> 3) : (uint32_t)(kWinBits / 8);
      const uint8_t *wb = reinterpret_cast<const uint8_t *>(win);
      uint8_t *o = dst + gbyte + (w0 >> 3);
      for (uint32_t i = t; i < nbytes; i += blockDim.x) o[i] = wb[i];
      __syncthreads();
      // carry the unfinished tail (partial byte, or the slack words) to the front of the window
      uint32_t c0 = 0, c1 = 0;
      if (last_win) {
        c0 = ((vend - w0) & 7) ? wb[nbytes] : 0;
      } else {
        c0 = win[kWinWords];
        c1 = win[kWinWords + 1];
      }
      __syncthreads();
      // only the words this window touched need clearing
      const int used = last_win ? (int)((vend - w0 + 31) >> 5) + 3 : kWinWords + 2;
      for (int i = t; i < min(used, kWinWords + 2); i += blockDim.x) win[i] = i == 0 ? c0 : (i == 1 ? c1 : 0u);
      __syncthreads();
      if (last_win) break;
    }
    gbits += piece_bits;
  }
  // final partial byte (its padding bits are zero here; k_huff_stale adds the stale ones)
  if (t == 0) {
    if (gbits & 7) dst[gbits >> 3] = (uint8_t)win[0];
    if (gbits != seg_bits[(size_t)item * hg.nseg + b]) atomicMax(err, 99);  // internal consistency
  }
}

// ---- K-pack (balanced) -----------------------------------------------------------------------
constexpr int kWin2Words = 4096;  // 16 KiB bit window + slack words
constexpr int kWin2Bits = kWin2Words * 32;

// Balanced item list as in k_huff_hist2; a thread takes EIGHT CONSECUTIVE items of a round of 2048,
// builds their tokens once ([zero-run token][literal code], usually < 16 bits per item) and keeps
// them in registers; one block scan of the per-thread bit totals gives its position, and the bits
// go into the window through a 64-bit register accumulator, one atomicOr per 32-bit WORD instead
// of up to three per token.  The window is flushed only when the next round would not fit.
constexpr int kP3Items = 8;
constexpr int kP3MinCtas = 5;  // 48 registers: five CTAs per SM (shared memory allows five) measured 7 % faster than four
constexpr int kP3Round = kTokThreads * kP3Items;

// zero run of z (1 <= z < kMaxRun) bytes -> token value and length; tab[s] = {code, len | lenx << 8}
__device__ __forceinline__ void run_token(const uint2 *tab, uint32_t z, uint64_t *tok, uint32_t *bits) {
  int sym = 260;
  uint32_t base = 279;
  if (z <= 278) sym = 259, base = 23;
  if (z <= 22) sym = 258, base = 7;
  if (z <= 6) sym = 257, base = 3;
  if (z <= 2) sym = z == 1 ? 0 : 256, base = z;
  const uint2 r = tab[sym];
  *tok = (uint64_t)r.x | ((uint64_t)(z - base) << (r.y & 255u));
  *bits = r.y >> 8;
}

// ORs n (<= 64) bits into the window at bit position pos (two slack words behind the window)
__device__ __forceinline__ void put64(uint32_t *win, uint32_t pos, uint64_t val, uint32_t n) {
  if (n == 0) return;
  const uint32_t word = pos >> 5, sh = pos & 31;
  const uint64_t v0 = val << sh;
  const uint32_t lo = (uint32_t)v0, mid = (uint32_t)(v0 >> 32), hi = sh ? (uint32_t)(val >> (64 - sh)) : 0u;
  if (lo) atomicOr(&win[word], lo);
  if (mid) atomicOr(&win[word + 1], mid);
  if (hi) atomicOr(&win[word + 2], hi);
}

// grid (nseg, n), block kTokThreads.  MIXED: see MixedHuff.
template <bool MIXED = false>
__global__ void __launch_bounds__(kTokThreads, kP3MinCtas)
    k_huff_pack3(const uint8_t *__restrict__ in, HuffGeom hg, const TreeOut *__restrict__ trees,
                 const uint32_t *__restrict__ seg_bits, const uint32_t *__restrict__ seg_pos,
                 const uint32_t *__restrict__ part_start, const uint32_t *__restrict__ sizes,
                 uint8_t *__restrict__ out, unsigned long long out_stride, int *err, ItemLists lists, MixedHuff mh = {}) {
  __shared__ uint32_t win[kWin2Words + 4];
  __shared__ uint2 s_tab[kSyms];
  __shared__ int s_last;
  __shared__ uint32_t ws[kTokWarps + 1];
  __shared__ uint32_t s_half;
  __shared__ __align__(16) uint32_t rows[kTokThreads * kRowWords];
  __shared__ __align__(16) unsigned short ipos[kTokPiece + 8];
  const int item = blockIdx.y, t = threadIdx.x;
  const int b = blockIdx.x / hg.nsub, part = blockIdx.x - b * hg.nsub;
  if (sizes[item] == 0) return;  // did not fit (k_huff_layout)
  const TreeOut *tr = trees + item;
  for (int s = t; s < kSyms; s += blockDim.x) {
    const uint32_t l = tr->len[s];
    s_tab[s] = make_uint2(tr->code[s], l | ((l + (uint32_t)sym_extra_bits(s)) << 8));
  }
  for (int i = t; i < kWin2Words + 4; i += blockDim.x) win[i] = 0;
  __syncthreads();
  HuffGeom ig = hg;  // this item's chunk
  if (MIXED && !(mixed_chunk(mh, item, ig) && b < ig.nseg)) return;  // (uniform)
  const uint8_t *seg0 = in + (size_t)item * hg.in_stride + (size_t)b * ig.seg_size;
  const int p0 = part * ig.sub_size, plen = min(ig.sub_size, ig.seg_size - p0);
  const uint8_t *seg = seg0 + p0;
  // this part's bits start at bit `first_bit` of the segment and end where the next part starts
  const size_t pidx = ((size_t)item * hg.nseg + b) * hg.nsub + part;
  const uint32_t first_bit = part_start[pidx];
  const uint32_t end_bit = part + 1 < hg.nsub ? part_start[pidx + 1] : seg_bits[(size_t)item * hg.nseg + b];
  uint8_t *dst = out + (size_t)item * out_stride + seg_pos[(size_t)item * hg.nseg + b] + (first_bit >> 3);
  bool first_shared = (first_bit & 7) != 0;  // byte 0 of dst also holds the last bits of the previous part
  const uint32_t full_bits = s_tab[260].y >> 8;  // one maximal run token
  const uint64_t full_tok = (uint64_t)s_tab[260].x | ((uint64_t)(kMaxRun - 279) << (s_tab[260].y & 255u));

  uint32_t carry = part ? zeros_before(seg0, p0, &s_last) : 0u;  // zeros of the run that is still open
  uint32_t gbyte = 0;                                            // complete bytes already written to dst
  uint32_t wfill = first_bit & 7;  // bits in the window; window bit 0 = bit 0 of byte gbyte
  // Writes the complete bytes of the window to dst and keeps the unfinished byte.  Uniform call.
  auto flush = [&]() {
    __syncthreads();
    const uint32_t nbytes = wfill >> 3;
    const uint8_t *wb = reinterpret_cast<const uint8_t *>(win);
    uint8_t *o = dst + gbyte;
    for (uint32_t i = t; i < nbytes; i += kTokThreads) {
      if (i == 0 && first_shared) atomic_or_byte(o, wb[0]);
      else o[i] = wb[i];
    }
    if (nbytes) first_shared = false;
    const uint32_t keep = (wfill & 7) ? wb[nbytes] : 0u;
    __syncthreads();
    const uint32_t used = min((wfill >> 5) + 4u, (uint32_t)(kWin2Words + 4));
    for (uint32_t i = t; i < used; i += kTokThreads) win[i] = i == 0 ? keep : 0u;
    __syncthreads();
    gbyte += nbytes;
    wfill &= 7;
  };
  // nfull maximal run tokens (16662 zeros each), cut greedily from the start of a run.  Uniform call.
  auto emit_full_runs = [&](uint32_t nfull) {
    while (nfull) {
      const uint32_t cap = ((uint32_t)kWin2Bits - wfill) / full_bits;
      if (cap == 0) {
        flush();
        continue;
      }
      const uint32_t n = min(nfull, cap);
      if (t == 0)
        for (uint32_t i = 0; i < n; ++i) put64(win, wfill + i * full_bits, full_tok, full_bits);
      wfill += n * full_bits;
      nfull -= n;
    }
  };

  uint8_t *ival = reinterpret_cast<uint8_t *>(rows);  // byte values of a stored list (the rows are not needed then)
  for (int base = 0; base < plen; base += kTokPiece) {
    PieceItems P;
    bool from_list = false;
    if (lists.pieces_per_part) {
      const size_t slot = item_slot(lists, hg, item, base / kTokPiece);
      const uint32_t cnt = lists.count[slot];
      if (cnt != kItemsNotStored) {
        // the list of k_huff_hist2: 16 / 8 bytes per thread and step, then one barrier
        from_list = true;
        const uint4 *gp = reinterpret_cast<const uint4 *>(lists.pos + slot * kItemCap);
        const uint2 *gv = reinterpret_cast<const uint2 *>(lists.val + slot * kItemCap);
        for (uint32_t i = t; i * 8 < cnt; i += kTokThreads) {
          reinterpret_cast<uint4 *>(ipos)[i] = __ldg(gp + i);
          reinterpret_cast<uint2 *>(ival)[i] = __ldg(gv + i);
        }
        __syncthreads();
        P.count = (int)cnt;
        P.len = min(kTokPiece, plen - base);
        P.zeros_in = carry;
        carry = cnt ? (uint32_t)(P.len - 1 - (int)ipos[cnt - 1]) : carry + (uint32_t)P.len;
      }
    }
    if (!from_list) carry = build_items(seg, plen, base, rows, ipos, ws, carry, &P);
    auto byte_of = [&](int k, int pos) -> uint32_t { return from_list ? (uint32_t)ival[k] : item_byte(rows, pos); };
    // a first gap of 16662 zeros or more: its maximal tokens go out first, the remainder stays with item 0
    uint32_t gap0_cut = 0;
    if (P.count > 0) {
      const uint32_t gap0 = (uint32_t)ipos[0] + P.zeros_in;
      if (gap0 >= (uint32_t)kMaxRun) {
        gap0_cut = (gap0 / kMaxRun) * kMaxRun;
        emit_full_runs(gap0 / kMaxRun);
      }
    }
    for (int r0 = 0; r0 < P.count; r0 += kP3Round) {
      const int k0 = r0 + t * kP3Items;
      const int m = min(max(P.count - k0, 0), kP3Items);
      uint64_t tok[kP3Items];
      uint32_t tl[kP3Items];
      uint32_t tbits = 0;
      bool wide = false;  // an item of more than 32 bits: this thread bypasses the accumulator
      if (m > 0) {
        const uint4 pv = *reinterpret_cast<const uint4 *>(ipos + k0);
        const uint32_t pw[4] = {pv.x, pv.y, pv.z, pv.w};
        int prev = k0 ? (int)ipos[k0 - 1] : -1;
#pragma unroll
        for (int j = 0; j < kP3Items; ++j) {
          tok[j] = 0;
          tl[j] = 0;
          if (j < m) {
            const int pos = (int)((pw[j >> 1] >> (16 * (j & 1))) & 0xffffu);
            uint32_t gap = (uint32_t)(pos - prev - 1);
            if (k0 + j == 0) gap += P.zeros_in - gap0_cut;
            prev = pos;
            const uint2 lr = s_tab[byte_of(k0 + j, pos)];
            uint64_t tk = lr.x;
            uint32_t l = lr.y & 255u;
            if (gap) {
              uint64_t rt;
              uint32_t rb;
              run_token(s_tab, gap, &rt, &rb);
              tk = rb + l <= 64 ? (rt | (tk << rb)) : rt;  // > 64 bits: the run token alone, literal re-read later
              l += rb;
            }
            wide |= l > 32;
            tok[j] = tk;
            tl[j] = l;
            tbits += l;
          }
        }
      }
      uint32_t total;
      const uint32_t tb = block_exscan_u32(tbits, ws, &total);
      if (wfill + total > (uint32_t)kWin2Bits) flush();
      // A round of incompressible data may not fit even the empty window: two halves then.
      const bool split = wfill + total > (uint32_t)kWin2Bits;
      if (split) {
        if (t == kTokThreads / 2) s_half = tb;
        __syncthreads();
      }
      const uint32_t half0 = split ? s_half : total;
      for (int hlf = 0; hlf < (split ? 2 : 1); ++hlf) {
        if (hlf == 1) flush();
        const bool mine = !split || (t >= kTokThreads / 2) == (hlf == 1);
        const uint32_t rel = hlf == 1 ? tb - half0 : tb;
        if (mine && m > 0) {
          uint32_t pos = wfill + rel;
          if (!wide) {
            uint32_t word = pos >> 5, fill = pos & 31;
            uint64_t acc = 0;
#pragma unroll
            for (int j = 0; j < kP3Items; ++j) {
              acc |= tok[j] << fill;  // tl <= 32 and fill < 32
              fill += tl[j];
              if (fill >= 32) {
                atomicOr(&win[word], (uint32_t)acc);
                acc >>= 32;
                fill -= 32;
                ++word;
              }
            }
            if ((uint32_t)acc) atomicOr(&win[word], (uint32_t)acc);
          } else {
#pragma unroll
            for (int j = 0; j < kP3Items; ++j) {
              if (j < m) {
                if (tl[j] <= 64) {
                  put64(win, pos, tok[j], tl[j]);
                } else {  // run token, then the literal
                  const uint2 lr = s_tab[byte_of(k0 + j, (int)ipos[k0 + j])];
                  const uint32_t rb = tl[j] - (lr.y & 255u);
                  put64(win, pos, tok[j], rb);
                  put64(win, pos + rb, lr.x, lr.y & 255u);
                }
                pos += tl[j];
              }
            }
          }
        }
        wfill += hlf == 1 ? total - half0 : half0;
      }
    }
    __syncthreads();  // rows / ipos are rewritten by the next piece
  }
  // the run still open at the segment end (an open run at the end of a part belongs to the next part)
  if (carry && part == hg.nsub - 1) {
    emit_full_runs(carry / kMaxRun);
    const uint32_t rest = carry % kMaxRun;
    if (rest) {
      uint64_t rt;
      uint32_t rb;
      run_token(s_tab, rest, &rt, &rb);
      if (wfill + rb > (uint32_t)kWin2Bits) flush();
      if (t == 0) put64(win, wfill, rt, rb);
      wfill += rb;
    }
  }
  flush();
  // final partial byte (its padding bits are zero here; k_huff_stale adds the stale ones)
  if (t == 0) {
    const uint32_t gbits = (first_bit & ~7u) + gbyte * 8u + wfill;
    if (wfill) {
      if (part + 1 < hg.nsub || first_shared) atomic_or_byte(dst + gbyte, win[0]);
      else dst[gbyte] = (uint8_t)win[0];
    }
    if (gbits != end_bit) atomicMax(err, 99);  // internal consistency
  }
}

// =================================================================================================
// Warp teams (v4) for framed chunks whose segments are not split into parts.  A CTA holds eight
// consecutive segments of one item, one warp per segment, and a warp synchronises with __syncwarp
// only: the block scans and barriers of every 8 KiB piece of k_huff_hist2 / k_huff_pack3 go away, and
// the item list of a segment is one contiguous list without piece boundaries.
// =================================================================================================
constexpr int kTeamWarps = 8;
constexpr int kTeamThreads = kTeamWarps * 32;
constexpr int kWalkStep = 32 * 16;  // bytes per warp step: 16 per lane

__device__ __forceinline__ uint4 load16(const uint8_t *__restrict__ seg, int seg_size, int off, bool aligned) {
  if (aligned && off + 16 <= seg_size) return __ldg(reinterpret_cast<const uint4 *>(seg + off));
  uint32_t w[4] = {0, 0, 0, 0};
#pragma unroll
  for (int k = 0; k < 16; ++k)
    if (off + k < seg_size) w[k >> 2] |= (uint32_t)seg[off + k] << (8 * (k & 3));
  return make_uint4(w[0], w[1], w[2], w[3]);
}

// Walks a segment in 512-byte warp steps and appends the position and value of every non-zero byte
// ("item") to a per-warp queue in shared memory: qpos[1 + k] / qval[1 + k] is item k of the queue,
// qpos[0] the position of the item before it (-1 at the segment start), so that the zero run in front
// of item k is qpos[1 + k] - qpos[k] - 1.  Whenever kRound items are queued, consume(k0, cnt, g0)
// takes items k0 .. k0 + cnt of the queue (g0: their index in the segment); the last call may take
// fewer.  Queues hold kRound + kWalkStep entries.  Returns the position of the segment's last item, or
// -1.  Warp-uniform call.
template <int kRound, class Consume>
__device__ __forceinline__ int warp_walk_items(const uint8_t *__restrict__ seg, int seg_size, int *qpos, uint8_t *qval,
                                               Consume &&consume) {
  const int lane = threadIdx.x & 31;
  const bool aligned = (reinterpret_cast<uintptr_t>(seg) & 15) == 0;
  if (lane == 0) qpos[0] = -1;
  __syncwarp();
  int qn = 0, g0 = 0;
  uint4 nxt = load16(seg, seg_size, 16 * lane, aligned);
  for (int base = 0; base < seg_size; base += kWalkStep) {
    const int off = base + 16 * lane;
    const uint4 w = nxt;
    nxt = load16(seg, seg_size, off + kWalkStep, aligned);  // (nothing past the segment end)
    uint32_t m = nonzero_nibble(w.x) | nonzero_nibble(w.y) << 4 | nonzero_nibble(w.z) << 8 | nonzero_nibble(w.w) << 12;
    const uint32_t c = __popc(m);
    uint32_t inc = c;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, inc, d);
      if (lane >= d) inc += t;
    }
    const int step_items = (int)__shfl_sync(0xffffffffu, inc, 31);
    if (step_items == 0) continue;
    int k = 1 + qn + (int)(inc - c);
    while (m) {
      const int j = __ffs(m) - 1;
      m &= m - 1;
      const uint32_t word = j < 4 ? w.x : (j < 8 ? w.y : (j < 12 ? w.z : w.w));
      qpos[k] = off + j;
      qval[k] = (uint8_t)(word >> (8 * (j & 3)));
      ++k;
    }
    qn += step_items;
    __syncwarp();
    if (qn >= kRound) {
      int done = 0;
      for (; qn - done >= kRound; done += kRound) consume(done, kRound, g0 + done);
      // the last consumed item and the rest move to the front (the ranges do not overlap: done >= kRound > rest)
      __syncwarp();
      for (int i = lane; i <= qn - done; i += 32) {
        qpos[i] = qpos[done + i];
        qval[i] = qval[done + i];
      }
      g0 += done;
      qn -= done;
      __syncwarp();
    }
  }
  if (qn) consume(0, qn, g0);
  return qpos[qn];
}

// Item list of a segment, handed from k_huff_hist4 to k_huff_pack4: the zero run in front of each item
// (u16) and its byte value, ItemLists::pieces_per_part * kItemCap entries per segment (the capacity of
// the per-piece lists of the same segment).  A segment with more items, or a run of 65536 zeros or
// more, is marked kItemsNotStored and the packer walks its planes again.
__device__ __forceinline__ size_t seg_list_base(const ItemLists &L, int nseg, int item, int b) {
  return ((size_t)item * nseg + b) * ((size_t)L.pieces_per_part * kItemCap);
}

// grid (ceil(nseg / 8), n), block 256: warp w codes segment 8 * blockIdx.x + w of item blockIdx.y.
// seghist: [n][nseg][261]; total: [n][261] (atomics).  MIXED: see MixedHuff.
template <bool MIXED = false>
__global__ void __launch_bounds__(kTeamThreads)
    k_huff_hist4(const uint8_t *__restrict__ in, HuffGeom hg, uint32_t *__restrict__ seghist, ItemLists lists,
                 uint32_t *__restrict__ total, MixedHuff mh = {}) {
  constexpr int kQ = 32 + kWalkStep;
  __shared__ uint32_t sh[kTeamWarps][kSyms];
  __shared__ int qpos_all[kTeamWarps][kQ];
  __shared__ uint8_t qval_all[kTeamWarps][kQ];
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31, item = blockIdx.y;
  const int b = blockIdx.x * kTeamWarps + wid;
  if (b >= hg.nseg) return;
  HuffGeom ig = hg;  // this item's chunk
  if (MIXED && !(mixed_chunk(mh, item, ig) && b < ig.nseg)) {  // idle segment: a zero histogram row
    for (int i = lane; i < kSyms; i += 32) seghist[((size_t)item * hg.nseg + b) * kSyms + i] = 0;
    return;
  }
  uint32_t *h = sh[wid];
  int *qpos = qpos_all[wid];
  uint8_t *qval = qval_all[wid];
  for (int i = lane; i < kSyms; i += 32) h[i] = 0;
  __syncwarp();
  const uint8_t *seg = in + (size_t)item * hg.in_stride + (size_t)b * ig.seg_size;
  const bool lists_on = lists.pieces_per_part != 0;
  const int cap = lists.pieces_per_part * kItemCap;
  unsigned short *lpos = lists_on ? lists.pos + seg_list_base(lists, hg.nseg, item, b) : nullptr;
  uint8_t *lval = lists_on ? lists.val + seg_list_base(lists, hg.nseg, item, b) : nullptr;
  bool long_gap = false;  // a run that the u16 list entry cannot hold
  auto run = [&](uint32_t z) {
    if (z >= (uint32_t)kMaxRun) {
      atomicAdd(&h[260], z / kMaxRun);
      z %= kMaxRun;
    }
    uint32_t ex;
    if (z) atomicAdd(&h[run_symbol(z, &ex)], 1u);
  };
  int nitems = 0;
  // one item per lane
  const int last = warp_walk_items<32>(seg, ig.seg_size, qpos, qval, [&](int k0, int cnt, int g0) {
    nitems = g0 + cnt;
    if (lane < cnt) {
      const int k = k0 + lane;
      const uint32_t gap = (uint32_t)(qpos[1 + k] - qpos[k] - 1), v = qval[1 + k];
      run(gap);
      atomicAdd(&h[v], 1u);
      long_gap |= gap > 0xffffu;
      if (lists_on && g0 + lane < cap) {
        lpos[g0 + lane] = (unsigned short)gap;
        lval[g0 + lane] = (uint8_t)v;
      }
    }
  });
  if (lane == 0) run((uint32_t)(ig.seg_size - 1 - last));  // the run still open at the segment end
  __syncwarp();
  if (lists_on) {
    const bool stored = nitems <= cap && !__any_sync(0xffffffffu, long_gap);
    if (lane == 0) lists.count[(size_t)item * hg.nseg + b] = stored ? (uint32_t)nitems : kItemsNotStored;
  }
  uint32_t *dst = seghist + ((size_t)item * hg.nseg + b) * kSyms;
  for (int i = lane; i < kSyms; i += 32) {
    const uint32_t v = h[i];
    dst[i] = v;
    if (total && v) atomicAdd(&total[(size_t)item * kSyms + i], v);
  }
}

// grid (ceil(nseg / 8), n), block 256: warp w packs segment 8 * blockIdx.x + w of item blockIdx.y.  Rounds of
// 32 lanes x 8 consecutive items in segment order; bit offsets from a warp scan; the bits go into a per-warp
// window in shared memory through a 64-bit accumulator (one atomicOr per word), and the warp writes the
// window out when the next round does not fit.
constexpr int kP4Items = 8;
constexpr int kP4Round = 32 * kP4Items;
constexpr int kWin4Words = 512;  // 2 KiB per warp (a q50 segment is ~6 KB)
constexpr int kWin4Bits = kWin4Words * 32;
constexpr int kP4Queue = kP4Round + kWalkStep;
constexpr int kP4MinCtas = 4;  // 64 registers, 49 KiB of shared memory per CTA
// dynamic shared memory: per warp a window, and a queue for the segments without a stored list
constexpr int kP4Smem = kTeamWarps * ((kWin4Words + 4) * 4 + kP4Queue * 5);

// MIXED: see MixedHuff.
template <bool MIXED = false>
__global__ void __launch_bounds__(kTeamThreads, kP4MinCtas)
    k_huff_pack4(const uint8_t *__restrict__ in, HuffGeom hg, const TreeOut *__restrict__ trees,
                 const uint32_t *__restrict__ seg_bits, const uint32_t *__restrict__ seg_pos,
                 const uint32_t *__restrict__ sizes, uint8_t *__restrict__ out, unsigned long long out_stride, int *err,
                 ItemLists lists, MixedHuff mh = {}) {
  extern __shared__ uint32_t p4_smem[];
  __shared__ uint2 s_tab[kSyms];
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31, item = blockIdx.y;
  if (sizes[item] == 0) return;  // did not fit (k_huff_layout)
  const TreeOut *tr = trees + item;
  for (int s = threadIdx.x; s < kSyms; s += blockDim.x) {
    const uint32_t l = tr->len[s];
    s_tab[s] = make_uint2(tr->code[s], l | ((l + (uint32_t)sym_extra_bits(s)) << 8));
  }
  __syncthreads();
  const int b = blockIdx.x * kTeamWarps + wid;
  if (b >= hg.nseg) return;
  HuffGeom ig = hg;  // this item's chunk
  if (MIXED && !(mixed_chunk(mh, item, ig) && b < ig.nseg)) return;
  uint32_t *win = p4_smem + wid * (kWin4Words + 4);
  int *qpos = reinterpret_cast<int *>(p4_smem + kTeamWarps * (kWin4Words + 4)) + wid * kP4Queue;
  uint8_t *qval = reinterpret_cast<uint8_t *>(p4_smem + kTeamWarps * (kWin4Words + 4 + kP4Queue)) + wid * kP4Queue;
  for (int i = lane; i < kWin4Words + 4; i += 32) win[i] = 0;
  __syncwarp();
  const uint8_t *seg = in + (size_t)item * hg.in_stride + (size_t)b * ig.seg_size;
  uint8_t *dst = out + (size_t)item * out_stride + seg_pos[(size_t)item * hg.nseg + b];
  const uint32_t full_bits = s_tab[260].y >> 8;  // one maximal run token
  const uint64_t full_tok = (uint64_t)s_tab[260].x | ((uint64_t)(kMaxRun - 279) << (s_tab[260].y & 255u));

  uint32_t gbyte = 0;  // complete bytes already written to dst
  uint32_t wfill = 0;  // bits in the window; window bit 0 = bit 0 of byte gbyte
  // Writes the complete bytes of the window to dst and keeps the unfinished byte.  Warp-uniform call.
  auto flush = [&]() {
    __syncwarp();
    const uint32_t nbytes = wfill >> 3;
    const uint8_t *wb = reinterpret_cast<const uint8_t *>(win);
    for (uint32_t i = lane; i < nbytes; i += 32) dst[gbyte + i] = wb[i];
    const uint32_t keep = (wfill & 7) ? wb[nbytes] : 0u;
    __syncwarp();
    const uint32_t used = min((wfill >> 5) + 4u, (uint32_t)(kWin4Words + 4));
    for (uint32_t i = lane; i < used; i += 32) win[i] = i == 0 ? keep : 0u;
    __syncwarp();
    gbyte += nbytes;
    wfill &= 7;
  };
  // Token by token, lane 0 writing: maximal runs, runs, literals that are out of the ordinary.  Uniform calls.
  auto put_uniform = [&](uint64_t v, uint32_t n) {
    if (wfill + n > (uint32_t)kWin4Bits) flush();
    if (lane == 0) put64(win, wfill, v, n);
    wfill += n;
  };
  auto run_uniform = [&](uint32_t z) {
    for (uint32_t nfull = z / kMaxRun; nfull;) {
      const uint32_t cap = ((uint32_t)kWin4Bits - wfill) / full_bits;
      if (cap == 0) {
        flush();
        continue;
      }
      const uint32_t n = min(nfull, cap);
      if (lane == 0)
        for (uint32_t i = 0; i < n; ++i) put64(win, wfill + i * full_bits, full_tok, full_bits);
      wfill += n * full_bits;
      nfull -= n;
    }
    const uint32_t rest = z % kMaxRun;
    if (rest) {
      uint64_t rt;
      uint32_t rb;
      run_token(s_tab, rest, &rt, &rb);
      put_uniform(rt, rb);
    }
  };
  // One round: lane i takes items 8i .. 8i + m - 1 of the round.  fetch8(gap, val) gives the zero run in
  // front of them and their byte values; fetch1(k, gap, val) item k of the round, for the rare paths (so
  // that the common one holds only the tokens in registers).
  auto round = [&](int m, auto &&fetch8, auto &&fetch1) {
    uint64_t tok[kP4Items];
    uint32_t tl[kP4Items];
    uint32_t tbits = 0;
    bool wide = false;  // an item of more than 32 bits: this lane bypasses the accumulator
    uint32_t gap[kP4Items], val[kP4Items];
    fetch8(gap, val);
#pragma unroll
    for (int j = 0; j < kP4Items; ++j) {
      tok[j] = 0;
      tl[j] = 0;
      if (j < m) {
        const uint2 lr = s_tab[val[j]];
        uint64_t tk = lr.x;
        uint32_t l = lr.y & 255u;
        const uint32_t nfull = gap[j] / kMaxRun, z = gap[j] - nfull * kMaxRun;
        if (z) {
          uint64_t rt;
          uint32_t rb;
          run_token(s_tab, z, &rt, &rb);
          tk = rt | (tk << rb);  // (only used when it fits 32 bits)
          l += rb;
        }
        wide |= l > 32 || nfull;
        l += nfull * full_bits;
        tok[j] = tk;
        tl[j] = l;
        tbits += l;
      }
    }
    uint32_t inc = tbits;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, inc, d);
      if (lane >= d) inc += t;
    }
    const uint32_t total = __shfl_sync(0xffffffffu, inc, 31);
    if (wfill + total > (uint32_t)kWin4Bits) flush();
    if (wfill + total > (uint32_t)kWin4Bits) {
      // does not fit even the empty window (long zero runs, or very long codes): item by item
      for (int L = 0; L < 32; ++L) {
        const int mL = __shfl_sync(0xffffffffu, m, L);
#pragma unroll
        for (int j = 0; j < mL; ++j) {
          uint32_t g, v;
          fetch1(kP4Items * L + j, g, v);
          run_uniform(g);
          put_uniform(s_tab[v].x, s_tab[v].y & 255u);
        }
      }
      return;
    }
    uint32_t pos = wfill + inc - tbits;
    if (!wide) {
      uint32_t word = pos >> 5, fill = pos & 31;
      uint64_t acc = 0;
#pragma unroll
      for (int j = 0; j < kP4Items; ++j) {
        acc |= tok[j] << fill;  // tl <= 32 and fill < 32
        fill += tl[j];
        if (fill >= 32) {
          atomicOr(&win[word], (uint32_t)acc);
          acc >>= 32;
          fill -= 32;
          ++word;
        }
      }
      if ((uint32_t)acc) atomicOr(&win[word], (uint32_t)acc);
    } else {
#pragma unroll
      for (int j = 0; j < kP4Items; ++j) {
        if (j < m) {
          uint32_t g, v;
          fetch1(kP4Items * lane + j, g, v);
          const uint32_t nfull = g / kMaxRun, z = g - nfull * kMaxRun;
          for (uint32_t f = 0; f < nfull; ++f, pos += full_bits) put64(win, pos, full_tok, full_bits);
          if (z) {
            uint64_t rt;
            uint32_t rb;
            run_token(s_tab, z, &rt, &rb);
            put64(win, pos, rt, rb);
            pos += rb;
          }
          const uint2 lr = s_tab[v];
          put64(win, pos, lr.x, lr.y & 255u);
          pos += lr.y & 255u;
        }
      }
    }
    wfill += total;
  };

  int last;  // position of the segment's last item
  const uint32_t cnt = lists.pieces_per_part ? lists.count[(size_t)item * hg.nseg + b] : kItemsNotStored;
  if (cnt != kItemsNotStored) {
    // the list of k_huff_hist4: 16 + 8 bytes per lane and round, the next round's loads in flight
    const size_t lb = seg_list_base(lists, hg.nseg, item, b);
    const uint4 *gp = reinterpret_cast<const uint4 *>(lists.pos + lb);
    const uint2 *gv = reinterpret_cast<const uint2 *>(lists.val + lb);
    uint32_t span = 0;  // bytes covered by this lane's items (run + literal)
    uint4 np = make_uint4(0, 0, 0, 0);
    uint2 nv = make_uint2(0, 0);
    if (kP4Items * lane < (int)cnt) np = __ldg(gp + lane), nv = __ldg(gv + lane);
    for (int r0 = 0; r0 < (int)cnt; r0 += kP4Round) {
      const int k0 = r0 + kP4Items * lane, m = min(max((int)cnt - k0, 0), kP4Items);
      const uint4 p = np;
      const uint2 v = nv;
      if (k0 + kP4Round < (int)cnt) np = __ldg(gp + (k0 + kP4Round) / kP4Items), nv = __ldg(gv + (k0 + kP4Round) / kP4Items);
      round(
          m,
          [&](uint32_t(&gap)[kP4Items], uint32_t(&val)[kP4Items]) {
            const uint32_t pw[4] = {p.x, p.y, p.z, p.w}, vw[2] = {v.x, v.y};
#pragma unroll
            for (int j = 0; j < kP4Items; ++j) {
              gap[j] = (pw[j >> 1] >> (16 * (j & 1))) & 0xffffu;
              val[j] = (vw[j >> 2] >> (8 * (j & 3))) & 0xffu;
              if (j < m) span += gap[j] + 1;
            }
          },
          [&](int k, uint32_t &g, uint32_t &val) {
            g = lists.pos[lb + r0 + k];
            val = lists.val[lb + r0 + k];
          });
    }
    last = (int)__reduce_add_sync(0xffffffffu, span) - 1;
  } else {
    // no list: the items again from the planes, with the walk of k_huff_hist4
    last = warp_walk_items<kP4Round>(seg, ig.seg_size, qpos, qval, [&](int k0, int n, int) {
      const int m = min(max(n - kP4Items * lane, 0), kP4Items);
      auto fetch1 = [&](int k, uint32_t &g, uint32_t &val) {
        g = (uint32_t)(qpos[1 + k0 + k] - qpos[k0 + k] - 1);
        val = qval[1 + k0 + k];
      };
      round(
          m,
          [&](uint32_t(&gap)[kP4Items], uint32_t(&val)[kP4Items]) {
#pragma unroll
            for (int j = 0; j < kP4Items; ++j) {
              gap[j] = 0;
              val[j] = 0;
              if (j < m) fetch1(kP4Items * lane + j, gap[j], val[j]);
            }
          },
          fetch1);
    });
  }
  run_uniform((uint32_t)(ig.seg_size - 1 - last));  // the run still open at the segment end
  flush();
  // final partial byte (its padding bits are zero here; k_huff_stale adds the stale ones)
  if (lane == 0) {
    if (wfill) dst[gbyte] = (uint8_t)win[0];
    if (gbyte * 8u + wfill != seg_bits[(size_t)item * hg.nseg + b]) atomicMax(err, 99);  // internal consistency
  }
}

// ---- K-stale ---------------------------------------------------------------------------------
// Padding bit p of segment b takes the value WRITTEN at bit p by the most recent earlier segment
// of the same chunk that is longer than p bits (else 0).  One thread per segment; the bit lengths of the
// block's segments and of the 1024 before them sit in shared memory (the walk back over earlier segments
// was a chain of dependent global loads; it rarely goes further, and then reads global memory again).
// grid (ceil(nseg / 256), n), block 256.
// MIXED (the FRES chunk of a mixed-geometry batch): nseg is the bounding segment count (the slot stride of the
// segment tables); item i has gi.rows segments.
constexpr int kStaleWindow = 1024;
template <bool MIXED = false>
__global__ void __launch_bounds__(256)
    k_huff_stale(int n, int nseg, const uint32_t *__restrict__ seg_bits, const uint32_t *__restrict__ seg_pos,
                 const uint32_t *__restrict__ sizes, uint8_t *__restrict__ out, unsigned long long out_stride,
                 MixedDims md = {}) {
  __shared__ uint32_t sb[kStaleWindow + 256];
  const int item = blockIdx.y, b0 = blockIdx.x * 256, b = b0 + (int)threadIdx.x;
  if (sizes[item] == 0) return;  // (uniform)
  const uint32_t *bits = seg_bits + (size_t)item * nseg;
  const uint32_t *pos = seg_pos + (size_t)item * nseg;
  if (MIXED) {
    Geom gi;
    image_geom(md, item, gi);  // (dims out of bounds: size 0 above)
    nseg = gi.rows;
    if (b0 >= nseg) return;  // (uniform)
  }
  const int w0 = max(0, b0 - kStaleWindow), w1 = min(nseg, b0 + 256);
  for (int i = threadIdx.x; i < w1 - w0; i += 256) sb[i] = bits[w0 + i];
  __syncthreads();
  if (b == 0 || b >= nseg) return;
  uint32_t lo = sb[b - w0];
  const uint32_t hi = (lo + 7) & ~7u;  // exclusive end of the padding
  if (lo == hi) return;
  uint8_t *base = out + (size_t)item * out_stride;
  const uint32_t byte_idx = lo >> 3;
  uint32_t add = 0;
  for (int e = b - 1; e >= 0 && lo < hi; --e) {
    const uint32_t le = e >= w0 ? sb[e - w0] : bits[e];
    if (le > lo) {
      const uint32_t upto = min(le, hi);  // positions [lo, upto) come from segment e
      const uint32_t mask = ((1u << (upto - (byte_idx << 3))) - 1u) & ~((1u << (lo - (byte_idx << 3))) - 1u);
      add |= base[pos[e] + byte_idx] & mask;
      lo = upto;
    }
  }
  if (add) base[pos[b] + byte_idx] |= (uint8_t)add;
}

}  // namespace himgcu

#endif  // HIMG_B200_HUFF_ENC_KERNELS_CUH_
