// RIFF container parsing + RLE/Huffman DECODE kernels (reference: decoder.cpp:144-272, :428-461,
// huffman_dec.cpp:152-418).  Every read is bounds-checked: hostile streams are rejected, never
// over-read (the reference's unchecked fast loop has undefined behaviour there).
//
//   k_dec_parse    one thread per image: RIFF/FRMT/LMAP/LRES/QCFG/FMAP/FRES walk + table recovery
//   k_dec_tree        one CTA per chunk: serialised tree -> packed nodes, single- and multi-token LUTs,
//                     second-level tables for codes longer than the LUT window
//   k_dec_segtab      one thread per chunk: walk the 2/4-byte segment headers
//   k_dec_stream_par  a team of threads per stream (warp per block-row segment / CTA / cluster of
//                     CTAs): subsequence-parallel, self-synchronising decode (see the kernel)
#ifndef HIMG_B200_HUFF_DEC_KERNELS_CUH_
#define HIMG_B200_HUFF_DEC_KERNELS_CUH_

#include <cooperative_groups.h>

#include "common.cuh"

namespace himgcu {

#ifndef HIMG_DEC_LUT_BITS
#define HIMG_DEC_LUT_BITS 11
#endif
constexpr int kLutBits = HIMG_DEC_LUT_BITS;
constexpr int kLutSize = 1 << kLutBits;

// Decode LUT entry (indexed by the next kLutBits stream bits, LSB first):
//   bits 0-7   literal byte (0 for zero-run tokens)
//   bits 8-12  code length in bits (0 only for a single-leaf tree in strict mode)
//   bits 13-16 number of extra bits that follow the code (0, 2, 4, 8 or 14)
//   bits 17-25 run base: output bytes = base + extra  (1 for literals)
//   bit 30     invalid slot (incomplete tree or symbol > 260)
//   bit 31     code longer than kLutBits: bits 0-15 hold the tree node reached after kLutBits bits
constexpr uint32_t kLutLong = 0x80000000u, kLutInvalid = 0x40000000u;
// Second level for codes longer than the window: every internal node at depth kLutBits gets a table
// of the next kSubBits bits (entries as above with the length counted from the window's end; a
// code longer than kLutBits + kSubBits keeps kLutLong | node and is finished by a tree walk).
constexpr int kSubBits = 5, kSubCap = 64;

__host__ __device__ inline uint32_t lut_entry(int sym, int len) {
  if (sym > 260) return kLutInvalid;
  uint32_t lit = 0, nx = 0, base = 1;
  if (sym <= 255) lit = (uint32_t)sym;
  else if (sym == 256) base = 2;
  else if (sym == 257) nx = 2, base = 3;
  else if (sym == 258) nx = 4, base = 7;
  else if (sym == 259) nx = 8, base = 23;
  else nx = 14, base = 279;
  return lit | ((uint32_t)len << 8) | (nx << 13) | (base << 17);
}

struct ChunkDesc {
  unsigned long long off;  // byte offset of the chunk payload inside the data buffer
  uint32_t size;
  uint32_t ok;
};

// Multi-token LUT entry (same index): every token that is completely determined by the 10 window
// bits, up to two non-zero literals.
// The last token of a group may be a zero run whose code lies in the window but whose extra bits do
// not: they are then read from the bit buffer ("tail").
//   x: bits 0-3 window bits consumed, 4-13 output bytes
//      produced (without the tail's extra value), 14-17 tail extra bits (0 = none), 18-27 offset of
//      the first non-zero literal
//   y: bits 0-7 first non-zero literal, 8-17 offset of the second, 18-25 its value, 26-27 number of
//      non-zero literals
// No token (x bits 0-3 = 0): x = kLutLong | node << 4 | (second-level table + 1) << 14 (the first code
// is longer than the window; node reached after kLutBits bits), kLutInvalid, or 0 (single-leaf tree).
struct __align__(16) DecTree {
  uint32_t lut[kLutSize];  // see lut_entry()
  uint2 lut2[kLutSize];
  uint32_t nodes[kMaxNodes + 1];  // leaf: 0x80000000 | symbol; internal: child0 | child1 << 16 (0xffff = none)
  uint32_t sub[kSubCap << kSubBits];
  int nnodes;
  int nsub;      // second-level tables in use
  int data_off;  // first byte after the (byte-aligned) tree
  int ok;
  int single;    // single-leaf tree
};

struct alignas(8) SegRef {
  uint32_t off;   // relative to the chunk payload
  uint32_t size;  // 0xffffffff = invalid
};

__device__ __forceinline__ uint32_t rd_u32(const uint8_t *p) {
  return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}

// Mapping function bytes -> unmap table (mapper.cpp:127-157) by the lanes of a warp (entry i sits at byte i while
// i <= single, at 1 + single + 2 (i - single - 1) after that).  A first byte above 127 -- where the
// reference writes past its table -- is rejected.  Uniform result.
__device__ __forceinline__ bool parse_mapfun_warp(const uint8_t *in, int size, int16_t *unmap, int lane) {
  if (size < 1) return false;
  const int single = in[0];
  if (single > 127 || 1 + single + 2 * (127 - single) != size) return false;
  if (lane == 0) unmap[0] = 0;
  for (int i = 1 + lane; i <= 127; i += 32) {
    uint32_t v;
    if (i <= single) {
      v = in[i];
    } else {
      const uint8_t *q = in + 1 + single + 2 * (i - single - 1);
      v = (uint32_t)q[0] | ((uint32_t)q[1] << 8);
    }
    const short sv = (short)(unsigned short)v;
    unmap[i] = sv;
    unmap[256 - i] = (short)(-sv);
    if (i == 127) unmap[128] = (short)(-sv);  // = unmap[129]
  }
  return true;
}

// grid: ceil(n / 4) x 128 threads; one WARP per image: lane 0 walks the RIFF chunk headers (a short chain of
// dependent loads), then the lanes parse the three tables side by side -- one thread doing it all was 125 us
// for a batch, whatever its size, and the first 26 us of every single-image decode.
// MIXED: the FRMT shape is checked against image i's dims of `md` (w, h are then unused), and dims that are < 1 or
// exceed the bounds make the image's status 2 (HIMGCU_ERR_ARG) and its chunks invalid.
template <bool MIXED = false>
__global__ void __launch_bounds__(128)
    k_dec_parse(const uint8_t *__restrict__ data, const unsigned long long *__restrict__ offsets,
                const uint32_t *__restrict__ sizes, int n, int w, int h, int nch,
                ChunkDesc *__restrict__ lres, ChunkDesc *__restrict__ fres,
                DecTables *__restrict__ tabs, int *__restrict__ status, MixedDims md = {}) {
  const int i = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (i >= n) return;
  bool bad_dims = false;
  if (MIXED) {
    Geom gi;
    bad_dims = !image_geom(md, i, gi);
    w = gi.w;
    h = gi.h;
  }
  const unsigned long long base = offsets[i];
  const uint8_t *p = data + base;
  const long long size = sizes[i];
  DecTables *T = tabs + i;
  // chunk offsets (relative to p) and sizes in file order: FRMT LMAP LRES QCFG FMAP FRES
  long long coff[6] = {0, 0, 0, 0, 0, 0};
  long long csz[6] = {-1, -1, -1, -1, -1, -1};
  int ok = 0;
  if (lane == 0) {
    ok = 1;
    if (MIXED && bad_dims) ok = 0;
    if (size < 12 || rd_u32(p) != 0x46464952u /*RIFF*/ || rd_u32(p + 8) != 0x474d4948u /*HIMG*/) ok = 0;
    if (ok && (long long)(int)rd_u32(p + 4) + 8 != size) ok = 0;
    long long idx = 12;
    const uint32_t want[6] = {0x544d5246u /*FRMT*/, 0x50414d4cu /*LMAP*/, 0x5345524cu /*LRES*/,
                              0x47464351u /*QCFG*/, 0x50414d46u /*FMAP*/, 0x53455246u /*FRES*/};
    for (int k = 0; k < 6 && ok; ++k) {
      for (;;) {  // FindRIFFChunk: unknown chunks are skipped (decoder.cpp:445-461)
        if (idx + 8 > size) {
          ok = 0;
          break;
        }
        const uint32_t cc = rd_u32(p + idx);
        const int sz = (int)rd_u32(p + idx + 4);
        idx += 8;
        if (sz < 0 || idx + sz > size) {
          ok = 0;
          break;
        }
        if (cc == want[k]) {
          coff[k] = idx;
          csz[k] = sz;
          idx += sz;
          break;
        }
        idx += sz;
      }
      // (the reference stops at the first chunk it cannot use: later chunks are not looked at)
      if (ok && k == 0) {
        const uint8_t *c = p + coff[0];
        if (csz[0] < 11 || c[0] != 1 || (int)rd_u32(c + 1) != w || (int)rd_u32(c + 5) != h || (int)c[9] != nch) ok = 0;
      }
    }
  }
  ok = __shfl_sync(0xffffffffu, ok, 0);
#pragma unroll
  for (int k = 0; k < 6; ++k) {
    coff[k] = __shfl_sync(0xffffffffu, coff[k], 0);
    csz[k] = __shfl_sync(0xffffffffu, csz[k], 0);
  }
  int ycbcr = 0;
  if (ok) {
    ycbcr = (p[coff[0] + 10] != 0 && nch >= 3) ? 1 : 0;
    if (!parse_mapfun_warp(p + coff[1], (int)csz[1], T->low_unmap, lane)) ok = 0;
    if (ok && csz[3] != (ycbcr ? 64 : 32)) ok = 0;
    if (ok) {
      const uint8_t *c = p + coff[3];
      const int q = lane;  // 32 bytes of luma shifts, 32 of chroma shifts: a byte pair per lane
      T->shift[0][2 * q] = c[q] >> 4;
      T->shift[0][2 * q + 1] = c[q] & 15;
      T->shift[1][2 * q] = ycbcr ? (c[32 + q] >> 4) : 0;
      T->shift[1][2 * q + 1] = ycbcr ? (c[32 + q] & 15) : 0;
    }
    if (ok && !parse_mapfun_warp(p + coff[4], (int)csz[4], T->full_unmap, lane)) ok = 0;
  }
  if (lane == 0) {
    T->ycbcr = ok ? ycbcr : 0;
    lres[i].off = base + (ok ? (unsigned long long)coff[2] : 0ull);
    lres[i].size = ok ? (uint32_t)csz[2] : 0u;
    lres[i].ok = ok ? 1u : 0u;
    fres[i].off = base + (ok ? (unsigned long long)coff[5] : 0ull);
    fres[i].size = ok ? (uint32_t)csz[5] : 0u;
    fres[i].ok = ok ? 1u : 0u;
    status[i] = MIXED && bad_dims ? 2 : (ok ? 0 : 1);
  }
}

// Chunk descriptors for the stage-level API (n equally strided chunks).
__global__ void k_dec_make_desc(unsigned long long stride, const uint32_t *__restrict__ sizes, int n,
                                ChunkDesc *__restrict__ cd, int *__restrict__ status) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  cd[i].off = (unsigned long long)i * stride;
  cd[i].size = sizes[i];
  cd[i].ok = 1;
  status[i] = 0;
}

// ---- tree recovery (huffman_dec.cpp:152-213) ---------------------------------------------------
constexpr int kDecTreeThreads = 256;

// grid (n, 1 or 2): blockIdx.y selects the chunk (cd0 / trees0 or cd1 / trees1), so that the two
// trees of an image are recovered side by side.
__global__ void __launch_bounds__(kDecTreeThreads)
    k_dec_tree(const uint8_t *__restrict__ data, const ChunkDesc *__restrict__ cd0, const ChunkDesc *__restrict__ cd1,
               int lenient, DecTree *__restrict__ trees0, DecTree *__restrict__ trees1, int *__restrict__ status) {
  const ChunkDesc *__restrict__ cd = blockIdx.y ? cd1 : cd0;
  DecTree *__restrict__ trees = blockIdx.y ? trees1 : trees0;
  __shared__ __align__(8) uint8_t raw[kTreeBytesMax + 16];
  __shared__ short ca[kMaxNodes], cb[kMaxNodes], nsym[kMaxNodes];
  __shared__ uint8_t depth[kMaxNodes];
  __shared__ int s_n, s_ok, s_bits;
  __shared__ uint32_t s_lut[kLutSize];   // the single-token LUT is built here (the multi-token LUT reads it back 2048 x ~4 times)
  __shared__ short stk[kMaxNodes + 2];   // branches whose right child is pending
  __shared__ short pslot[kMaxNodes];     // 2 * parent + (right child ? 1 : 0); -1 for the root
  __shared__ short anc[kMaxNodes];     // ancestor at depth kLutBits (-1: none)
  __shared__ uint8_t subc[kMaxNodes];  // code bits kLutBits .. kLutBits + kSubBits - 1
  __shared__ short xsub[kMaxNodes];    // second-level table of a depth-kLutBits node
  __shared__ int s_nsub;
  const int item = blockIdx.x, t = threadIdx.x;
  DecTree *out = trees + item;
  const ChunkDesc d = cd[item];
  const int avail = d.ok ? (int)min((uint32_t)kTreeBytesMax, d.size) : 0;
  for (int i = t; i < kTreeBytesMax + 16; i += blockDim.x) raw[i] = i < avail ? data[d.off + i] : 0;
  for (int i = t; i < kMaxNodes; i += blockDim.x) ca[i] = cb[i] = nsym[i] = -1;
  __syncthreads();
  if (t == 0) {
    // Pre-order walk of the serialised tree (leaf = bit 1 + 9-bit symbol, branch = bit 0) by ONE thread: a
    // lone thread issues a dependent instruction every few cycles, so the walk only records the STRUCTURE
    // (symbol, slot in the parent; a branch pushes itself for its right child, a leaf pops), with the bits
    // in a 64-bit register window.  Depths, codes and LUT ancestors follow in parallel below.
    // (Round 1 carried all of it through five stack arrays: 60 us for a 261-leaf tree.)
    int n = 0, ok = d.ok ? 1 : 0, sp = 0, bit = 0;
    const int nbits = avail * 8;
    const uint32_t *raw32 = reinterpret_cast<const uint32_t *>(raw);
    unsigned long long buf = (unsigned long long)raw32[0] | ((unsigned long long)raw32[1] << 32);
    int nb = 64, widx = 2, slot = -1;
    s_nsub = 0;
    bool more = ok != 0;
    while (more) {
      if (n >= kMaxNodes) {
        ok = 0;
        break;
      }
      const int k = n++;
      pslot[k] = (short)slot;
      if (bit + 1 > nbits) {
        ok = 0;
        break;
      }
      if (nb < 32) {  // (the array is padded with zero words: reading past the tree is harmless)
        buf |= (unsigned long long)raw32[widx++] << nb;
        nb += 32;
      }
      const int leaf = (int)(buf & 1u);
      buf >>= 1;
      --nb;
      ++bit;
      if (leaf) {
        if (bit + 9 > nbits) {
          ok = 0;
          break;
        }
        nsym[k] = (short)(buf & 511u);
        buf >>= 9;
        nb -= 9;
        bit += 9;
        if (sp == 0) more = false;
        else slot = stk[--sp];
      } else {
        stk[sp++] = (short)(k * 2 + 1);
        slot = k * 2;
      }
    }
    s_n = n;
    s_ok = ok;
    s_bits = bit;
  }
  __syncthreads();
  // Child links, then depth / code / sub-code / LUT ancestor of every node by a walk UP its parent chain
  // (a few dozen dependent shared-memory loads per node, all nodes at once, no barrier): the bits of the path
  // arrive deepest first, so shifting them in from the right leaves bit i of the code = branch taken at depth i.
  if (s_ok) {
    const int nn = s_n;
    for (int k = t; k < nn; k += blockDim.x) {
      int dlen = 0, cur = k;
      uint32_t acc = 0;
      for (int sl = pslot[cur]; sl >= 0; sl = pslot[cur]) {
        acc = (acc << 1) | (uint32_t)(sl & 1);
        cur = sl >> 1;
        ++dlen;
      }
      const int sl0 = pslot[k];
      if (sl0 >= 0) {
        if (sl0 & 1) cb[sl0 >> 1] = (short)k;
        else ca[sl0 >> 1] = (short)k;
      }
      depth[k] = (uint8_t)min(dlen, 255);
      subc[k] = (uint8_t)((acc >> kLutBits) & ((1u << kSubBits) - 1u));
      int a = -1;  // the ancestor at depth kLutBits starts the sub-code of everything below it
      if (dlen > kLutBits) {
        a = k;
        for (int up = dlen - kLutBits; up > 0; --up) a = pslot[a] >> 1;
      }
      anc[k] = (short)a;
    }
  }
  __syncthreads();
  const int n = s_n;
  if (!s_ok) {
    if (t == 0) {
      out->ok = 0;
      out->nnodes = 0;
      out->nsub = 0;
      out->data_off = 0;
      out->single = 0;
      atomicMax(&status[item], 1);
    }
    return;
  }
  const bool single = n == 1;
  for (int k = t; k < n; k += blockDim.x)
    out->nodes[k] = nsym[k] >= 0 ? (0x80000000u | (uint32_t)nsym[k])
                                 : (((uint32_t)ca[k] & 0xffffu) | (((uint32_t)cb[k] & 0xffffu) << 16));
  // single-token LUT: every window value walks down from the root (at most kLutBits steps); a leaf on the way
  // fills the entry, an internal node at depth kLutBits marks a longer code
  for (int p = t; p < kLutSize; p += blockDim.x) {
    int node = 0, pos = 0;
    uint32_t e = kLutInvalid;
    for (;;) {
      const int sy = nsym[node];
      if (sy >= 0) {
        // The reference's decoder consumes ZERO bits per symbol for a single-leaf tree
        // (huffman_dec.cpp:178-188) although its encoder wrote one; lenient mode consumes it.
        e = lut_entry(sy, (single && lenient) ? 1 : pos);
        break;
      }
      if (pos == kLutBits) {
        e = kLutLong | (uint32_t)node;
        break;
      }
      const int child = ((p >> pos) & 1) ? cb[node] : ca[node];
      if (child < 0) break;
      node = child;
      ++pos;
    }
    s_lut[p] = e;
  }
  if (t == 0) {
    out->ok = 1;
    out->nnodes = n;
    out->data_off = (s_bits + 7) >> 3;
    out->single = single ? 1 : 0;
  }
  // second-level tables of the internal nodes at depth kLutBits
  for (int i = t; i < (kSubCap << kSubBits); i += blockDim.x) out->sub[i] = kLutInvalid;
  for (int k = t; k < n; k += blockDim.x) {
    xsub[k] = -1;
    if (nsym[k] < 0 && depth[k] == kLutBits) {
      const int si = atomicAdd(&s_nsub, 1);
      if (si < kSubCap) xsub[k] = (short)si;
    }
  }
  __syncthreads();
  for (int k = t; k < n; k += blockDim.x) {
    const int d = (int)depth[k] - kLutBits;
    if (d < 1 || d > kSubBits || anc[k] < 0 || xsub[anc[k]] < 0) continue;
    uint32_t *tab = out->sub + ((int)xsub[anc[k]] << kSubBits);
    if (nsym[k] >= 0) {
      const uint32_t e = lut_entry(nsym[k], d);
      for (uint32_t i = 0; i < (1u << (kSubBits - d)); ++i) tab[(i << d) | subc[k]] = e;
    } else if (d == kSubBits) {
      tab[subc[k]] = kLutLong | (uint32_t)k;
    }
  }
  if (t == 0) out->nsub = min(s_nsub, kSubCap);
  __syncthreads();  // the single-token LUT (shared memory) and out->sub are complete
  for (int i = t; i < kLutSize; i += blockDim.x) out->lut[i] = s_lut[i];
  for (int p = t; p < kLutSize; p += blockDim.x) {
    int pos = 0, bytes = 0, nlit = 0, tail = 0;
    uint32_t off[2] = {0, 0}, lit[2] = {0, 0}, first = 0;
    while (!single && pos < kLutBits) {
      const uint32_t e = s_lut[(uint32_t)p >> pos];
      if (e & (kLutLong | kLutInvalid)) {
        if (pos == 0) {
          first = kLutInvalid;
          if (!(e & kLutInvalid)) {
            const int node = (int)(e & 0xffffu);
            first = kLutLong | ((uint32_t)node << 4) | ((uint32_t)(xsub[node] + 1) << 14);
          }
        }
        break;
      }
      const int len = (int)((e >> 8) & 31u), nx = (int)((e >> 13) & 15u);
      if (len == 0 || len > kLutBits - pos) break;  // the code is not determined by the window bits
      if (len + nx > kLutBits - pos) {              // zero run with its extra bits beyond the window
        bytes += (int)((e >> 17) & 511u);
        pos += len;
        tail = nx;
        break;
      }
      const uint32_t l = e & 255u;
      if (l) {
        if (nlit == 2) break;
        off[nlit] = (uint32_t)bytes;
        lit[nlit] = l;
        ++nlit;
      }
      bytes += (int)((e >> 17) & 511u) + (int)(((uint32_t)p >> (pos + len)) & ((1u << nx) - 1u));
      pos += len + nx;
    }
    out->lut2[p] = make_uint2(first | (uint32_t)pos | ((uint32_t)bytes << 4) | ((uint32_t)tail << 14) | (off[0] << 18),
                              lit[0] | (off[1] << 8) | (lit[1] << 18) | ((uint32_t)nlit << 26));
  }
}

// ---- segment table (huffman_dec.cpp:215-251) ---------------------------------------------------
// One thread per chunk.  mode: 0 = unframed chunk decoded as ONE stream (LRES, Uncompress);
// 1 = framed chunk of nseg block rows (FRES, UncompressBlock).
//
// The headers form a chain (each one sits behind the previous payload): ~0.3 us per segment, 100-350 us
// for the 270-1024 block rows of a single 4K / 8K image.  With PUBLISH the walk runs INSIDE the stream
// decode kernel (its first CTA) and releases every entry as soon as it is known; the decoding CTAs
// acquire theirs, so the decode of the first rows overlaps the rest of the walk.  Entries start as
// kSegNotReady (host memset) and always end up valid or invalid (0xffffffff).
constexpr uint32_t kSegNotReady = 0xfefefefeu;
// A segment (framed or not) of this many packed bytes or more is rejected.  No valid stream has one (a block row codes
// to fewer than 46 * 2^26 bits, see shape_ok), and the bound keeps PBits' 32-bit bit positions (8 * size) exact and
// every size clear of kSegNotReady on corrupt streams.
constexpr uint32_t kMaxSegPacked = 1u << 29;

// An entry is ONE aligned 8-byte word (offset | size << 32): a single store publishes it and a single
// load takes it, no fence (a release store per entry tripled the time of the walk).
static_assert(sizeof(SegRef) == 8, "SegRef is published as one 64-bit word");
template <bool PUBLISH>
__device__ __forceinline__ void seg_store(SegRef *s, uint32_t off, uint32_t size) {
  if (PUBLISH) {
    *reinterpret_cast<volatile unsigned long long *>(s) = (unsigned long long)off | ((unsigned long long)size << 32);
  } else {
    s->off = off;
    s->size = size;
  }
}
__device__ __forceinline__ SegRef seg_acquire(const SegRef *s) {
  SegRef r;
  for (;;) {
    const unsigned long long v = *reinterpret_cast<const volatile unsigned long long *>(s);
    r.off = (uint32_t)v;
    r.size = (uint32_t)(v >> 32);
    if (r.size != kSegNotReady) break;
    __nanosleep(500);
  }
  return r;
}

template <bool PUBLISH>
__device__ void segtab_walk(const uint8_t *__restrict__ data, const ChunkDesc d, const DecTree *__restrict__ T, int nseg,
                            int seg_size, int mode, int lenient, SegRef *__restrict__ S, int *__restrict__ status_i) {
  int done = 0;  // entries stored so far; on every exit the remaining ones become invalid
  auto fail = [&]() {
    for (int b = done; b < nseg; ++b) seg_store<PUBLISH>(S + b, 0, 0xffffffffu);
    atomicMax(status_i, 1);
  };
  if (!d.ok || !T->ok) return fail();
  const uint32_t start = (uint32_t)T->data_off;
  if (mode == 0) {
    // HuffmanDec(in, size, 0): block size = packed size => never framed; an empty payload can
    // only produce an empty output (huffman_dec.cpp:278-279).
    if (start >= d.size || d.size - start >= kMaxSegPacked) return fail();
    seg_store<PUBLISH>(S, start, d.size - start);
    done = 1;
    for (int b = done; b < nseg; ++b) seg_store<PUBLISH>(S + b, 0, 0xffffffffu);
    return;
  }
  // The reference decides framing by comparing the UNPACKED block size with the PACKED chunk size
  // (huffman_dec.cpp:217-218, SURVEY A.4-6); the encoder framed iff there is more than one segment.
  const bool framed = lenient ? (nseg > 1) : ((uint32_t)seg_size < d.size);
  if (!framed) {
    if (!lenient || start >= d.size) return fail();  // UncompressBlock refuses unframed data (:265)
    if (d.size - start >= kMaxSegPacked) return fail();
    seg_store<PUBLISH>(S, start, d.size - start);
    done = 1;
    for (int b = done; b < nseg; ++b) seg_store<PUBLISH>(S + b, 0, 0xffffffffu);
    return;
  }
  const uint8_t *p = data + d.off;
  uint32_t pos = start;
  for (int b = 0; b < nseg; ++b) {
    if (pos + 2 > d.size) return fail();
    uint32_t sz = (uint32_t)p[pos] | ((uint32_t)p[pos + 1] << 8);
    pos += 2;
    if (sz & 0x8000u) {
      if (pos + 2 > d.size) return fail();
      sz = (sz & 0x7fffu) | (((uint32_t)p[pos] | ((uint32_t)p[pos + 1] << 8)) << 15);
      pos += 2;
    }
    if ((unsigned long long)pos + sz > d.size || sz >= kMaxSegPacked) return fail();
    seg_store<PUBLISH>(S + b, pos, sz);
    done = b + 1;
    pos += sz;
  }
}

__global__ void k_dec_segtab(const uint8_t *__restrict__ data, const ChunkDesc *__restrict__ cd,
                             const DecTree *__restrict__ trees, int n, int nseg, int seg_size, int mode,
                             int lenient, SegRef *__restrict__ segs, int *__restrict__ status) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  segtab_walk<false>(data, cd[i], trees + i, nseg, seg_size, mode, lenient, segs + (size_t)i * nseg, status + i);
}

// Whole-image FRES segment table of a mixed-geometry batch: image i's header chain is walked for its own gi.rows
// segments of gi.seg bytes (so the framing decision is the image's own), into a table of `stride` (the bounding
// geometry's rows) entries per image.  Entries past gi.rows are left alone: k_dec_stream_par<..., kMixWhole> never
// reads them.  A separate kernel, so that k_dec_segtab keeps its code.
__global__ void k_dec_segtab_mixed(const uint8_t *__restrict__ data, const ChunkDesc *__restrict__ cd,
                                   const DecTree *__restrict__ trees, int n, int stride, int lenient,
                                   SegRef *__restrict__ segs, int *__restrict__ status, MixedDims md) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Geom gi;
  image_geom(md, i, gi);  // (dims out of bounds: the chunk is invalid, and the walk only marks entry 0 invalid)
  segtab_walk<false>(data, cd[i], trees + i, gi.rows, gi.seg, 1, lenient, segs + (size_t)i * stride, status + i);
}

// Region decode (framed FRES chunk): the segment table of the block rows r0 = y / 8 .. r1 = (y + rh - 1) / 8 that
// image i's rectangle touches, compacted to kr entries per image: entry k is row min(r0 + k, r1), so a rectangle
// that touches fewer than kr rows decodes its last row again instead of needing a "skip" entry.  The header
// chain is walked only to r1 (into the scratch table `full` [n][rows]; the walk has no end-of-chunk check, so
// these entries are those of a whole-image walk), and at least to row 1 of a multi-row image so that the lenient
// framing decision ("more than one segment") is the whole image's.  An origin that puts the rectangle outside
// the image makes the image's status 2 (HIMGCU_ERR_ARG) and all its entries invalid.
// MIXED: g is the bounding geometry (the stride of `full`); image i's header chain and origin are those of its own
// geometry from `md`, and dims out of bounds are treated as an origin outside the image.
template <bool MIXED = false>
__global__ void k_dec_segtab_region(const uint8_t *__restrict__ data, const ChunkDesc *__restrict__ cd,
                                    const DecTree *__restrict__ trees, int n, Geom g, int lenient,
                                    const int32_t *__restrict__ origins, int rw, int rh, int kr,
                                    SegRef *__restrict__ full, SegRef *__restrict__ segs, int *__restrict__ status,
                                    MixedDims md = {}) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  SegRef *S = segs + (size_t)i * kr;
  Geom gi = g;
  const bool dims_ok = !MIXED || image_geom(md, i, gi);
  int x, y;
  if (!dims_ok || !region_origin(origins, i, gi, rw, rh, x, y)) {
    for (int k = 0; k < kr; ++k) seg_store<false>(S + k, 0, 0xffffffffu);
    atomicMax(status + i, 2);
    return;
  }
  const int r0 = y >> 3, r1 = (y + rh - 1) >> 3;
  SegRef *F = full + (size_t)i * g.rows;
  segtab_walk<false>(data, cd[i], trees + i, gi.rows > 1 ? max(r1 + 1, 2) : 1, gi.seg, 1, lenient, F, status + i);
  for (int k = 0; k < kr; ++k) S[k] = F[min(r0 + k, r1)];
}

// ---- subsequence-parallel stream decode ---------------------------------------------------------
// A team of threads (one CTA) decodes ONE stream.  The bit stream is cut into equal subsequences;
// thread t starts decoding at a guessed position (the subsequence boundary, usually in the middle
// of a code word).  Huffman codes self-synchronise: after a few symbols a wrongly started decoder
// falls onto true code-word boundaries.  Rounds of "take the end position of the previous thread
// as my start" are repeated until nothing changes (thread 0 is right from the start, so round r
// fixes at least thread r; in practice 2-3 rounds).  Output offsets are a prefix sum of the
// per-thread byte counts, then every thread decodes its subsequence once more and writes.
struct PBits {
  const uint32_t *w;  // 4-byte aligned base at or below the stream start
  int last_word;      // last word index that holds a valid byte (-1: empty stream)
  uint32_t widx;
  uint32_t nxt;       // word widx, fetched one refill ahead so the load latency is off the critical path
  uint64_t buf;
  int nb;
  uint32_t pos;  // stream-relative bit position of buf bit 0
  __device__ __forceinline__ uint32_t ld(uint32_t i) const { return (int)i <= last_word ? __ldg(w + i) : 0u; }
  __device__ __forceinline__ void seek(const uint8_t *base, uint32_t nbytes, uint32_t bitpos) {
    const uintptr_t a = reinterpret_cast<uintptr_t>(base);
    const uint32_t boff = (uint32_t)(a & 3) * 8;
    w = reinterpret_cast<const uint32_t *>(a & ~(uintptr_t)3);
    last_word = nbytes ? (int)((boff + 8 * nbytes - 1) >> 5) : -1;
    const uint32_t ap = boff + bitpos;
    widx = ap >> 5;
    const uint32_t w0 = ld(widx), w1 = ld(widx + 1);
    widx += 2;
    nxt = ld(widx);
    buf = (((uint64_t)w1 << 32) | w0) >> (ap & 31);
    nb = 64 - (int)(ap & 31);
    pos = bitpos;
  }
  __device__ __forceinline__ void refill() {
    // select-based: lanes of a warp refill at different times, a branch here diverges constantly
    const bool r = nb <= 32;
    buf |= r ? (uint64_t)nxt << (nb & 63) : 0ull;
    nb += r ? 32 : 0;
    widx += r ? 1u : 0u;
    if (r) nxt = ld(widx);
  }
  __device__ __forceinline__ void consume(int n) {
    buf >>= n;
    nb -= n;
    pos += (uint32_t)n;
  }
};

// Decodes one token.  Returns the number of output bytes it stands for (1 for a literal, the run
// length for a zero-run token) or -1 on an invalid code; *lit receives the literal byte (0 for
// runs).  After refill() at least 33 bits are buffered: enough for a kLutBits-bit code + 14 extra bits.
// Finishes a token whose symbol is known: extra bits, run length.  Returns the output bytes.
__device__ __forceinline__ int finish_token(PBits &b, uint32_t e, int *lit) {
  b.consume((int)((e >> 8) & 31u));
  const int nx = (int)((e >> 13) & 15u);
  const int z = (int)((e >> 17) & 511u) + (int)((uint32_t)b.buf & ((1u << nx) - 1u));
  b.consume(nx);
  *lit = (int)(e & 255u);
  return z;
}
// Token whose code is longer than the LUT window: walk the tree from `node` (reached after kLutBits
// bits).  Returns the output bytes or -1.
__device__ __forceinline__ int decode_long(PBits &b, const uint32_t *nodes, int node, int *lit) {
  b.consume(kLutBits);
  uint32_t w = nodes[node];
  int guard = 0;
  while (!(w & 0x80000000u)) {
    b.refill();
    const uint32_t child = (b.buf & 1u) ? (w >> 16) : (w & 0xffffu);
    b.consume(1);
    if (child >= (uint32_t)kMaxNodes || ++guard > kMaxNodes) return -1;
    w = nodes[child];
  }
  const uint32_t e = lut_entry((int)(w & 0xffffu), 0);
  if (e & kLutInvalid) return -1;
  b.refill();
  return finish_token(b, e, lit);
}
// Same with the second-level table of the node (g = the multi-token LUT word of the window): one
// more lookup resolves codes of up to kLutBits + kSubBits bits; longer ones walk the tree.
__device__ __forceinline__ int decode_long2(PBits &b, const uint32_t *nodes, const uint32_t *sub, uint32_t g, int *lit) {
  const uint32_t si = (g >> 14) & 0xffu;
  if (si) {
    const uint32_t e = sub[((si - 1u) << kSubBits) + ((uint32_t)(b.buf >> kLutBits) & ((1u << kSubBits) - 1u))];
    if (!(e & (kLutLong | kLutInvalid))) {
      b.consume(kLutBits);
      return finish_token(b, e, lit);  // >= 33 bits were buffered: 11 + 5 + 14 fit
    }
  }
  return decode_long(b, nodes, (int)((g >> 4) & 0x3ffu), lit);
}
__device__ __forceinline__ int decode_token(PBits &b, const uint32_t *lut, const uint32_t *nodes, int *lit) {
  b.refill();
  const uint32_t e = __ldg(lut + ((uint32_t)b.buf & (kLutSize - 1)));
  if (e & (kLutLong | kLutInvalid)) {
    if (e & kLutInvalid) return -1;
    return decode_long(b, nodes, (int)(e & 0xffffu), lit);
  }
  return finish_token(b, e, lit);
}

constexpr uint32_t kPosInvalid = 0xffffffffu;
constexpr int kParFresThreads = 32;   // team per block-row segment
constexpr int kParLresThreads = 256;  // team for the single unframed LRES stream
constexpr int kParMaxTeam = 1024;

constexpr int kParWarpTeams = 8;  // WARP_TEAMS: streams (one warp each) per CTA

// WARP_TEAMS = false: grid (nseg, n), block TEAM (multiple of 32, <= 1024): one CTA per stream.
// WARP_TEAMS = true:  grid (ceil(nseg / 8), n), block 256: a warp per stream, eight consecutive
//   streams of the same image per CTA.  They share the image's LUT and tree in shared memory (1 KiB
//   of shared memory per stream instead of 12 KiB, so the kernel leaves room for CTAs of other
//   streams' kernels) and synchronise with __syncwarp only.
// CL > 1 (with WARP_TEAMS = false): grid (nseg * CL, n) launched as thread-block CLUSTERS of CL CTAs:
//   one team of CL * blockDim.x threads spread over CL SMs decodes one stream.  End positions,
//   flags and scan totals are exchanged through distributed shared memory, team barriers are
//   cluster barriers.  This is what a single large image needs: its low-res chunk is ONE stream,
//   and one CTA (one SM) was the whole machine for it.
// MIX (mixed-geometry batches, one CTA per stream or warp teams, no inline walk): the output size of a stream is
//   its image's own (from `md`): the low-res chunk (kMixLres) or a block row (kMixFres, kMixWhole); out_seg is unused.
//   kMixWhole (whole-image decode): nseg is the bounding geometry's rows, and block rows b >= gi.rows of an image
//   are idle (no status, nothing written): a CTA whose streams all lie past them exits before staging the tree.
constexpr int kMixLres = 1, kMixFres = 2, kMixWhole = 3;
template <bool WARP_TEAMS, int CL = 1, int MIX = 0>
__global__ void k_dec_stream_par(const uint8_t *__restrict__ data, const ChunkDesc *__restrict__ cd,
                                 const DecTree *__restrict__ trees, SegRef *__restrict__ segs, int nseg,
                                 int out_seg, uint8_t *__restrict__ out, unsigned long long out_stride,
                                 int *__restrict__ status, int inline_walk = 0, int lenient = 0, MixedDims md = {}) {
  __shared__ __align__(16) uint2 lut2[kLutSize];  // the single-token LUT stays in global memory (rare path)
  __shared__ uint32_t s_nodes[kMaxNodes + 1];
  __shared__ uint32_t s_sub[kSubCap << kSubBits];
  __shared__ uint32_t s_end_all[WARP_TEAMS ? 32 * kParWarpTeams : kParMaxTeam];
  __shared__ uint32_t ws[33];
  __shared__ int s_flags[3 * (WARP_TEAMS ? kParWarpTeams : 1)];
  __shared__ uint32_t s_tot;
  // one 32-byte output line per lane (word w of lane l at [warp][w][l]: conflict-free); CTAs of more
  // than eight warps (wide teams for a few large streams) write their literals directly
  __shared__ uint32_t s_line[kParWarpTeams * 8 * 32];
  static_assert(!(WARP_TEAMS && CL > 1), "clusters are for the one-stream-per-team variant");
  static_assert(MIX == 0 || CL == 1, "mixed geometry has no cluster decode");
  namespace cg = cooperative_groups;
  const int item = blockIdx.y;
  int mix_rows = 0;  // kMixWhole: block rows of the item's image
  if (MIX) {  // (an image with dims out of bounds has an invalid chunk: its tree is not ok and nothing is written)
    Geom gi;
    image_geom(md, item, gi);
    out_seg = MIX == kMixLres ? gi.lres_size : gi.seg;
    inline_walk = 0;
    mix_rows = gi.rows;
  }
  // inline_walk (one CTA per stream only): CTA 0 of every item walks the segment headers of the framed
  // chunk and publishes the table (see segtab_walk); the stream of CTA x is segment x - 1
  if (!WARP_TEAMS && CL == 1 && inline_walk && blockIdx.x == 0) {
    if (threadIdx.x == 0)
      segtab_walk<true>(data, cd[item], trees + item, nseg, out_seg, 1, lenient, segs + (size_t)item * nseg, status + item);
    return;
  }
  const int rank = CL > 1 ? (int)cg::this_cluster().block_rank() : 0;
  const int tm = WARP_TEAMS ? (int)(threadIdx.x >> 5) : 0;  // team inside the CTA
  const int lt = WARP_TEAMS ? (int)(threadIdx.x & 31) : (int)threadIdx.x;  // index inside this CTA's share of the team
  const int t = lt + rank * (int)blockDim.x, team = WARP_TEAMS ? 32 : CL * (int)blockDim.x;
  const int b = WARP_TEAMS ? (int)blockIdx.x * kParWarpTeams + tm
                           : (CL == 1 && inline_walk ? (int)blockIdx.x - 1 : (int)blockIdx.x / CL);
  auto tsync = [] {
    if (WARP_TEAMS) __syncwarp();
    else if (CL > 1) cg::this_cluster().sync();
    else __syncthreads();
  };
  // OR of a per-CTA flag over the cluster (after a team barrier; ends with one, so the flag may be
  // reused and a CTA may exit)
  auto team_or = [&](int *flag) -> bool {
    bool any = *flag != 0;
    if (CL > 1) {
      for (int r = 0; r < CL; ++r) any |= *cg::this_cluster().map_shared_rank(flag, r) != 0;
      cg::this_cluster().sync();
    }
    return any;
  };
  if (MIX == kMixWhole && (WARP_TEAMS ? (int)blockIdx.x * kParWarpTeams : b) >= mix_rows) return;  // (the whole CTA)
  const DecTree *T = trees + item;
  if (T->ok) {  // the whole CTA stages the image's LUT and tree
    const uint4 *l2 = reinterpret_cast<const uint4 *>(T->lut2);
#pragma unroll 4
    for (int i = threadIdx.x; i < kLutSize / 2; i += blockDim.x) reinterpret_cast<uint4 *>(lut2)[i] = __ldg(l2 + i);
    const int nn = T->nnodes;
    for (int i = threadIdx.x; i < nn; i += blockDim.x) s_nodes[i] = T->nodes[i];
    const int ns = T->nsub << kSubBits;
    for (int i = threadIdx.x; i < ns; i += blockDim.x) s_sub[i] = T->sub[i];
  }
  __syncthreads();
  if (WARP_TEAMS && b >= nseg) return;
  if (MIX == kMixWhole && b >= mix_rows) return;
  SegRef sr;
  if (!WARP_TEAMS && CL == 1 && inline_walk) {
    // ONE thread polls (a whole grid of polling threads slowed the walker's own dependent loads down)
    __shared__ SegRef s_sr;
    if (threadIdx.x == 0) s_sr = seg_acquire(segs + (size_t)item * nseg + b);
    __syncthreads();
    sr = s_sr;
  } else {
    sr = segs[(size_t)item * nseg + b];
  }
  if (!T->ok || sr.size == 0xffffffffu || sr.size == 0) {  // an empty stream cannot produce out_seg > 0 bytes
    if (t == 0) atomicMax(&status[item], 1);
    return;
  }
  uint32_t *s_end = s_end_all + 32 * tm;
  int &s_changed = s_flags[3 * tm], &s_bad = s_flags[3 * tm + 1], &s_final = s_flags[3 * tm + 2];
  const uint32_t *SN = s_nodes;
  const uint32_t *lut = T->lut;
  if (lt == 0) s_bad = 0, s_final = -1;
  int *final_pos = CL > 1 ? cg::this_cluster().map_shared_rank(&s_final, 0) : &s_final;  // lives in CTA 0
  tsync();
  const uint8_t *src = data + cd[item].off + sr.off;
  uint8_t *o = out + (size_t)item * out_stride + (size_t)b * out_seg;
  const uint32_t total_bits = sr.size * 8u;

  // The segment is zero-filled cooperatively (coalesced stores); the write pass then only stores
  // the non-zero literals -- three out of four coefficient bytes are zeros at quality 50.
  const bool al16 = ((reinterpret_cast<uintptr_t>(o) | (uintptr_t)out_seg) & 15) == 0;
  {
    if (al16) {
      for (int i = t; i < (out_seg >> 4); i += team) reinterpret_cast<uint4 *>(o)[i] = make_uint4(0, 0, 0, 0);
    } else {
      for (int i = t; i < out_seg; i += team) o[i] = 0;
    }
  }
  tsync();

  if (T->single) {
    // Single-leaf tree: every token has the same code (0 bits for the reference decoder, 1 bit in
    // lenient mode, see k_dec_tree); nothing to parallelise.
    if (t == 0) {
      PBits br;
      br.seek(src, sr.size, 0);
      int n = 0;
      bool ok = true;
      while (n < out_seg) {
        int lit;
        const int z = decode_token(br, lut, SN, &lit);
        if (z < 0 || br.pos > total_bits || n + z > out_seg) {
          ok = false;
          break;
        }
        if (lit) o[n] = (uint8_t)lit;
        n += z;
      }
      if (ok) ok = br.pos > 8u * (sr.size - 1) && br.pos <= total_bits;
      if (!ok) atomicMax(&status[item], 1);
    }
    return;
  }

  // ---- phase 1: synchronise.  Thread t owns the tokens that START in [start_t, end_t).
  uint32_t sub = (total_bits + team - 1) / team;
  sub = max((sub + 31u) & ~31u, 128u);
  const uint32_t bound_lo = min((uint32_t)t * sub, total_bits);        // nominal start
  const uint32_t bound_hi = min((uint32_t)(t + 1) * sub, total_bits);  // tokens starting here belong to t+1
  const bool has_work = bound_lo < total_bits;
  uint32_t start = bound_lo, endpos = kPosInvalid, count = 0;
  bool dirty = has_work;
  // Checkpoints of my previous decode: position of the first decode step at or after bound_lo + 64,
  // 128, 256, 512 bits and the bytes counted before it.  A re-decode from a corrected start that
  // lands on one of them continues exactly like the previous decode, so it stops there and
  // splices the counts: the second round costs a few dozen bits instead of the whole subsequence.
  constexpr int kCp = 4;
  uint32_t cpp[kCp], cpc[kCp];
#pragma unroll
  for (int i = 0; i < kCp; ++i) cpp[i] = kPosInvalid, cpc[i] = 0;
  for (int round = 0; round <= team; ++round) {
    if (dirty) {
      PBits br;
      br.seek(src, sr.size, start);
      uint32_t cnt = 0, next_ms = bound_lo + 64u;
      int mi = 0;
      bool ok = true, spliced = false;
      while (br.pos < bound_hi) {
        if (br.pos >= next_ms) {
          uint32_t old_pos = kPosInvalid, old_cnt = 0;
#pragma unroll
          for (int i = 0; i < kCp; ++i)
            if (i == mi) {
              old_pos = cpp[i];
              old_cnt = cpc[i];
              cpp[i] = br.pos;
              cpc[i] = cnt;
            }
          if (old_pos == br.pos) {
            const uint32_t delta = cnt - old_cnt;
#pragma unroll
            for (int i = 0; i < kCp; ++i)
              if (i > mi) cpc[i] += delta;
            count += delta;  // endpos: as before
            spliced = true;
            break;
          }
          ++mi;
          next_ms = mi < kCp ? bound_lo + (64u << mi) : 0xffffffffu;
        }
        br.refill();
        // A group that STARTS in my range is mine even if its later tokens start beyond bound_hi: the
        // next thread begins wherever I end.  Only the last bits of the stream (where the padding
        // would be parsed as tokens) go through the single-token path.
        if (br.pos + kLutBits + 14 <= total_bits) {
          const uint32_t g = lut2[(uint32_t)br.buf & (kLutSize - 1)].x;
          if (g & 15u) {
            const int nb = (int)(g & 15u), nx = (int)((g >> 14) & 15u);
            cnt += ((g >> 4) & 1023u) + ((uint32_t)(br.buf >> nb) & ((1u << nx) - 1u));
            br.consume(nb + nx);
            continue;
          }
          if (g & kLutLong) {  // code longer than the window: no second table lookup
            int lit;
            const int z = decode_long2(br, SN, s_sub, g, &lit);
            if (z < 0 || br.pos > total_bits) {
              ok = false;
              break;
            }
            cnt += (uint32_t)z;
            continue;
          }
        }
        int lit;
        const int z = decode_token(br, lut, SN, &lit);
        if (z < 0 || br.pos > total_bits) {
          ok = false;
          break;
        }
        cnt += (uint32_t)z;
      }
      if (!spliced) {
        count = cnt;
        // the last subsequence may run into the (possibly non-zero) padding bits: that is not an error
        endpos = ok ? br.pos : (bound_hi == total_bits ? total_bits : kPosInvalid);
#pragma unroll
        for (int i = 0; i < kCp; ++i)
          if (i >= mi) cpp[i] = kPosInvalid;
      }
    }
    s_end[lt] = has_work ? endpos : kPosInvalid;
    if (lt == 0) s_changed = 0;
    tsync();
    dirty = false;
    if (has_work && t > 0) {
      const uint32_t prev = (CL == 1 || lt > 0) ? s_end[lt - 1]
                                                : cg::this_cluster().map_shared_rank(s_end, rank - 1)[blockDim.x - 1];
      // a start beyond my own range means the previous thread's token swallowed my subsequence
      if (prev != kPosInvalid && prev != start) {
        start = prev;
        dirty = start < bound_hi || bound_hi == total_bits;
        if (!dirty) {
          count = 0;
          endpos = start;  // nothing starts in my range: pass the position through
#pragma unroll
          for (int i = 0; i < kCp; ++i) cpp[i] = kPosInvalid;
        }
        s_changed = 1;
      }
    }
    tsync();
    if (!team_or(&s_changed)) break;
    if (CL == 1) tsync();  // (team_or ends with a barrier when the team spans CTAs)
  }

  // ---- output offsets
  uint32_t off;
  if (WARP_TEAMS) {
    const uint32_t v = has_work ? count : 0u;
    uint32_t inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t u = __shfl_up_sync(0xffffffffu, inc, d);
      if (t >= d) inc += u;
    }
    off = inc - v;
  } else {
    uint32_t total;
    off = block_exscan_u32(has_work ? count : 0u, ws, &total);
    if (CL > 1) {  // add the totals of the CTAs before mine
      if (lt == 0) s_tot = total;
      cg::this_cluster().sync();
      for (int r = 0; r < rank; ++r) off += *cg::this_cluster().map_shared_rank(&s_tot, r);
    }
  }
  // threads whose output lies inside the segment must have decoded cleanly
  if (has_work && off < (uint32_t)out_seg && endpos == kPosInvalid) s_bad = 1;
  tsync();
  if (team_or(&s_bad)) {
    if (t == 0) atomicMax(&status[item], 1);
    return;
  }

  // ---- phase 2: decode again and write the non-zero literals
  // One byte store per literal makes one 32-byte L2 write transaction per literal: the kernel was bound
  // by that, not by instructions.  A lane therefore collects the literals of the 32-byte lines that
  // lie completely inside its own output range in a shared-memory line and writes each line once
  // (two 16-byte stores, zeros included); only its first and last, shared, lines take byte stores.
  if (has_work && off < (uint32_t)out_seg && start < total_bits) {
    PBits br;
    br.seek(src, sr.size, start);
    int n = (int)off;
    bool ok = true;
    const bool buffered = (reinterpret_cast<uintptr_t>(o) & 15) == 0 && blockDim.x <= 32 * kParWarpTeams;
    uint32_t *line = s_line + (buffered ? (threadIdx.x >> 5) * 256 + (threadIdx.x & 31) : 0);
    const int line_lo = buffered ? (int)((off + 31u) >> 5) : 0x7fffffff;
    const int line_hi = (int)(min(off + count, (uint32_t)out_seg) >> 5);
    int cur = -1;
    if (buffered) {
#pragma unroll
      for (int k = 0; k < 8; ++k) line[k * 32] = 0;
    }
    auto flush_line = [&]() {
      if (cur >= 0) {
        uint32_t w[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          w[k] = line[k * 32];
          line[k * 32] = 0;
        }
        uint4 *d = reinterpret_cast<uint4 *>(o + (size_t)cur * 32);
        d[0] = make_uint4(w[0], w[1], w[2], w[3]);
        d[1] = make_uint4(w[4], w[5], w[6], w[7]);
      }
    };
    auto put = [&](int idx, uint32_t v) {
      const int ln = idx >> 5;
      if (ln >= line_lo && ln < line_hi) {
        if (ln != cur) {
          flush_line();
          cur = ln;
        }
        reinterpret_cast<uint8_t *>(line + ((idx >> 2) & 7) * 32)[idx & 3] = (uint8_t)v;
      } else {
        o[idx] = (uint8_t)v;
      }
    };
    while (br.pos < bound_hi && n < out_seg) {
      br.refill();
      uint32_t long_g = 0;
      if (br.pos + kLutBits + 14 <= total_bits) {  // same rule as in phase 1
        const uint2 g = lut2[(uint32_t)br.buf & (kLutSize - 1)];
        const int nb = (int)(g.x & 15u), nx = (int)((g.x >> 14) & 15u);
        const int gb = (int)((g.x >> 4) & 1023u) + (int)((uint32_t)(br.buf >> nb) & ((1u << nx) - 1u));
        if (nb && n + gb <= out_seg) {  // the whole group lies inside the segment
          if (g.y >> 26) {
            put(n + (int)((g.x >> 18) & 1023u), g.y);
            if ((g.y >> 26) > 1) put(n + (int)((g.y >> 8) & 1023u), g.y >> 18);
          }
          br.consume(nb + nx);
          n += gb;
          if (n == out_seg) *final_pos = (int)br.pos;
          continue;
        }
        if (!nb && (g.x & kLutLong)) long_g = g.x;
      }
      int lit;
      const int z = long_g ? decode_long2(br, SN, s_sub, long_g, &lit) : decode_token(br, lut, SN, &lit);
      if (z < 0 || br.pos > total_bits || n + z > out_seg) {
        ok = false;  // a zero run that overshoots the segment is an error (huffman_dec.cpp:352)
        break;
      }
      if (lit) put(n, (uint32_t)lit);
      n += z;
      if (n == out_seg) *final_pos = (int)br.pos;
    }
    flush_line();
    if (!ok) s_bad = 1;
  }
  tsync();
  const bool any_bad = team_or(&s_bad);
  if (t == 0) {
    // complete output, and the read position inside the last byte (BitStream::AtTheEnd)
    const bool ok = !any_bad && s_final >= 0 && (uint32_t)s_final > 8u * (sr.size - 1) && (uint32_t)s_final <= total_bits;
    if (!ok) atomicMax(&status[item], 1);
  }
}

}  // namespace himgcu

#endif  // HIMG_B200_HUFF_DEC_KERNELS_CUH_
