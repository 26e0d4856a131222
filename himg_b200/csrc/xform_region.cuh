// K-inv of a region decode: the inverse transform of the blocks a rectangle [x, x + rw) x [y, y + rh) of an image
// touches, with only the rectangle's pixels stored, tightly packed: pixel (Y, X) of the image goes to
// (Y - y) * rw * nch + (X - x) * nch of the image's output.  The coefficient planes are COMPACT, kr segments per image
// (see k_dec_segtab_region): slot k holds block row min(r0 + k, r1), r0 = y / 8, r1 = (y + rh - 1) / 8; a slot past r1
// is a repeat and is skipped.  The low-res image R is the whole image's, read at the real block row and column, so
// the corner and edge clamps of the interpolation are those of the image, not of the rectangle.
//
//   k_inverse_region4  fast path (nch 1 / 3, cols % 16 == 0): k_inverse4's lane pairs and warp tiles over the
//                      flattened (slot, block pair) space of the staged columns, clipped stores (Inv4StoreClip)
//   k_inverse_region   every other shape and force_generic: one block per thread in int32, as k_inverse, with a
//                      runtime channel count (colour map on channels 0-2)
#ifndef HIMG_B200_XFORM_REGION_CUH_
#define HIMG_B200_XFORM_REGION_CUH_

#include "common.cuh"
#include "xform_inv4.cuh"
#include "xform_kernels.cuh"

namespace himgcu {

// Pixel row y of a block pair, clipped to the rectangle.  The pair's 16 * NCH bytes of a row are one run in the
// output that starts at any byte alignment (the rectangle's origin and width are arbitrary), and only the bytes
// [b0, b1) of the run lie inside the rectangle.  The run is realigned with funnel shifts into the 4-byte words of
// the output: whole words inside the rectangle are 32-bit stores, the (at most two) words shared with a
// neighbouring pair and the words at the rectangle's left and right edges are byte stores.  A run that is whole
// and 16-byte aligned (a rectangle at x % 16 == 0 whose row bytes are a multiple of 16) is stored as k_inverse4
// stores it.
template <int NCH>
struct Inv4StoreClip {
  uint8_t *row0;       // byte 0 of the pair's pixel row 0 in the output (may lie outside the rectangle)
  long long row_bytes; // rw * NCH
  int y0, rh;          // pixel row 0 of the pair is row y0 of the rectangle
  int b0, b1;          // bytes of a run inside the rectangle
  __device__ __forceinline__ void operator()(int y, const uint32_t (&wa)[2 * NCH], const uint32_t (&wb)[2 * NCH]) const {
    if (y0 + y < 0 || y0 + y >= rh) return;
    constexpr int K = 4 * NCH;  // words of a run
    uint32_t W[K];
#pragma unroll
    for (int m = 0; m < 2 * NCH; ++m) {
      W[m] = wa[m];
      W[2 * NCH + m] = wb[m];
    }
    const uintptr_t addr = reinterpret_cast<uintptr_t>(row0) + (uintptr_t)((long long)y * row_bytes);
    if (b0 == 0 && b1 == 16 * NCH && (addr & 15) == 0) {
      uint4 *dst = reinterpret_cast<uint4 *>(addr);
#pragma unroll
      for (int k = 0; k < NCH; ++k) dst[k] = make_uint4(W[4 * k], W[4 * k + 1], W[4 * k + 2], W[4 * k + 3]);
      return;
    }
    const int a = (int)(addr & 3);
    uint8_t *base = reinterpret_cast<uint8_t *>(addr - (uintptr_t)a);
#pragma unroll
    for (int j = 0; j <= K; ++j) {
      const int s = 4 * j - a;  // run byte at the output word's byte 0
      const uint32_t v = __funnelshift_rc(j > 0 ? W[j - 1] : 0u, j < K ? W[j] : 0u, 8 * (4 - a));
      if (s >= b0 && s + 4 <= b1) {
        *reinterpret_cast<uint32_t *>(base + 4 * j) = v;
      } else {
#pragma unroll
        for (int t = 0; t < 4; ++t)
          if (s + t >= b0 && s + t < b1) base[4 * j + t] = (uint8_t)(v >> (8 * t));
      }
    }
  }
};

// Block pairs of a compact slot staged by k_inverse_region4 for a rectangle of width rw: the columns from the
// 16-block boundary at or below x / 8 (16-byte aligned cp.async sources) to (x + rw - 1) / 8, for the worst x, in
// whole 16-byte chunks (8 pairs), at most the image's.
inline int region_span_pairs(int rw, int cols) {
  const int kb = (rw + 14) / 8;  // block columns a rectangle of width rw can touch
  const int span = 8 * ((kb + 15 + 15) / 16);
  return span < cols / 2 ? span : cols / 2;
}

// grid (ceil(kr * span / TP), 1, n), block TP, dynamic smem as k_inverse4.  A CTA owns TP consecutive elements of
// the image's flattened [kr][span] space of block pairs; pairs outside the image or the rectangle and repeated
// slots are computed on whatever the tile holds and not stored.
template <int NCH, int TP>
__global__ void __launch_bounds__(TP, NCH == 1 ? 3 : 2)
    k_inverse_region4(const uint8_t *__restrict__ planes, const uint8_t *__restrict__ R, Geom g,
                      const InvTables *__restrict__ tabs, unsigned long long tab_stride, const int32_t *__restrict__ origins,
                      int rw, int rh, int kr, int span, uint8_t *__restrict__ pixels, uint32_t one) {
  extern __shared__ __align__(128) uint8_t sPl[];
  constexpr int PITCH = 2 * TP, CPR = TP / 8;
  static_assert(TP % 32 == 0 && TP == 8 * CPR, "a CTA is 8 groups of one thread per chunk of a tile row");
  uint8_t *sDq = sPl + NCH * 64 * PITCH;
  uint32_t *sTab = reinterpret_cast<uint32_t *>(sDq + kInvSlots * 256 * 2);
  const int item = blockIdx.z;
  int x, y;
  if (!region_origin(origins, item, g, rw, rh, x, y)) return;  // (the whole CTA)
  const int t = threadIdx.x;
  const int r0 = y >> 3, r1 = (y + rh - 1) >> 3;
  const int u0 = (x >> 3) & ~15, ul = x >> 3, ur = (x + rw - 1) >> 3;
  const int f0 = blockIdx.x * TP, nact = min(TP, kr * span - f0);
  const uint8_t *ipl = planes + (size_t)item * kr * g.seg;
  const InvTables *T = reinterpret_cast<const InvTables *>(reinterpret_cast<const char *>(tabs) + (size_t)item * tab_stride);
  {
    const uint4 *tsrc = reinterpret_cast<const uint4 *>(T);
    for (int i = t; i < kInvTableBytes / 16; i += TP) cp_async16(sDq + 16 * i, tsrc + i);
    // a chunk = 8 pairs of one slot (span % 8 == 0), inside the image or wholly outside it (cols % 16 == 0)
    const int cq = t % CPR, rt = t / CPR, e = f0 + 8 * cq;
    const int s = e / span, u = u0 + 2 * (e - s * span);
    if (8 * cq < nact && u < g.cols) {
      const uint8_t *src = ipl + (size_t)s * g.seg + u + (size_t)rt * g.cols;
      uint8_t *dst = sPl + rt * PITCH + cq * 16;
      const size_t rstep = (size_t)8 * g.cols;
#pragma unroll 8
      for (int i = 0; i < NCH * 8; ++i) {
        cp_async16(dst + i * 8 * PITCH, src);
        src += rstep;
      }
    }
  }
  const int e = f0 + t, s = e / span;
  int u = u0 + 2 * (e - s * span);
  const bool active = t < nact && r0 + s <= r1 && u < g.cols && u + 1 >= ul && u <= ur;
  if (!active) u = u0;  // (corner loads inside the image)
  const int v = min(r0 + s, r1);
  uint32_t top[NCH], bot[NCH];
  inv4_corners<NCH>(R, item, g, v, u, top, bot);
  const int X0 = 8 * u - x;  // rectangle column of the pair's first pixel
  const Inv4StoreClip<NCH> store{pixels + (size_t)item * rw * rh * NCH + ((long long)(8 * v - y) * rw + X0) * NCH,
                                 (long long)rw * NCH, 8 * v - y, rh, max(0, -X0) * NCH, min(16, rw - X0) * NCH};
  const int pre = T->pre, tab_bias = T->bias;
  const bool overflow = T->overflow != 0;
  const bool ycbcr = T->ycbcr != 0;
  cp_async_wait_all();
  __syncthreads();
  inv4_compute<NCH, PITCH, Inv4StoreClip<NCH>>(sPl + 2 * t, sDq, sTab, pre, tab_bias, overflow, ycbcr, active, top, bot, store,
                                               one);
}

// grid (ceil(kb / kTile), kr, n), block kTile (kb = (rw + 14) / 8 block columns): thread = block column x / 8 + i of
// compact slot blockIdx.y.  Same arithmetic as k_inverse.
// MIXED: g is the bounding geometry, which sets the slot strides (kr * g.seg bytes of planes and nch * rows * cols
// bytes of R per image); image item's planes (kr segments of its own size), low-res image, corners and origin check
// use its own geometry from `md`.  An image with dims out of bounds is not written.
template <bool MIXED = false>
__global__ void __launch_bounds__(kTile)
    k_inverse_region(const uint8_t *__restrict__ planes, const uint8_t *__restrict__ R, Geom g,
                     const DecTables *__restrict__ tabs, unsigned long long tab_stride, const int32_t *__restrict__ origins,
                     int rw, int rh, int kr, uint8_t *__restrict__ pixels, MixedDims md = {}) {
  __shared__ int16_t sUn[256];
  __shared__ uint8_t sShift[2][64];
  __shared__ uint32_t sOut[3][kTile][17];  // channels 0-2 of a thread's block (the colour map needs all three)
  const int item = blockIdx.z, slot = blockIdx.y;
  Geom gi = g;  // the image's geometry
  if (MIXED && !image_geom(md, item, gi)) return;
  int x, y;
  if (!region_origin(origins, item, gi, rw, rh, x, y)) return;  // (the whole CTA)
  const int v = (y >> 3) + slot;
  if (v > (y + rh - 1) >> 3) return;  // a repeated slot
  const DecTables *T = reinterpret_cast<const DecTables *>(reinterpret_cast<const char *>(tabs) + (size_t)item * tab_stride);
  for (int i = threadIdx.x; i < 256; i += blockDim.x) sUn[i] = T->full_unmap[i];
  for (int i = threadIdx.x; i < 128; i += blockDim.x) sShift[i >> 6][i & 63] = T->shift[i >> 6][i & 63];
  const int nch = g.nch;
  const bool ycbcr = T->ycbcr != 0 && nch >= 3;
  __syncthreads();
  const int u = (x >> 3) + blockIdx.x * kTile + threadIdx.x;
  if (u > (x + rw - 1) >> 3) return;
  const uint8_t *seg = MIXED ? planes + (size_t)item * kr * g.seg + (size_t)slot * gi.seg : planes + ((size_t)item * kr + slot) * g.seg;
  uint8_t *img = pixels + (size_t)item * rw * rh * nch;
  // pixels of the block inside the rectangle: rows [ya, yb), columns [xa, xb) of the block
  const int ya = max(0, y - 8 * v), yb = min(8, y + rh - 8 * v), xa = max(0, x - 8 * u), xb = min(8, x + rw - 8 * u);
  auto out = [&](int yy, int i) { return img + ((size_t)(8 * v + yy - y) * rw + (8 * u + i - x)) * nch; };
  const int ngroup = min(nch, 3);
#pragma unroll 1
  for (int c = 0; c < nch; ++c) {
    int xv[64];
    const uint8_t *src = seg + (size_t)c * gi.cols * 64 + u;
    const uint8_t *sh = sShift[(ycbcr && (c == 1 || c == 2)) ? 1 : 0];
#pragma unroll
    for (int j = 0; j < 64; ++j) xv[j] = (int)(short)(sUn[__ldg(src + (size_t)scan_pos(j) * gi.cols)] * (1 << sh[j]));
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      wht8(xv[r * 8 + 0], xv[r * 8 + 1], xv[r * 8 + 2], xv[r * 8 + 3], xv[r * 8 + 4], xv[r * 8 + 5], xv[r * 8 + 6], xv[r * 8 + 7]);
#pragma unroll
      for (int i = 0; i < 8; ++i) xv[r * 8 + i] >>= 3;
    }
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      wht8(xv[q], xv[8 + q], xv[16 + q], xv[24 + q], xv[32 + q], xv[40 + q], xv[48 + q], xv[56 + q]);
#pragma unroll
      for (int i = 0; i < 8; ++i) xv[i * 8 + q] >>= 3;
    }
    {
      const LowCorners k =
          load_corners(MIXED ? R + (size_t)item * nch * g.rows * g.cols + (size_t)c * gi.rows * gi.cols : R + ((size_t)item * nch + c) * g.rows * g.cols,
                       gi, u, v);
      int lf[9], rt[9];
      nine(k.x11, k.x21, lf);
      nine(k.x12, k.x22, rt);
#pragma unroll
      for (int yy = 0; yy < 8; ++yy) {
        int tl[9];
        nine(lf[yy], rt[yy], tl);
#pragma unroll
        for (int i = 0; i < 8; ++i) xv[yy * 8 + i] = clamp255((int)(short)(xv[yy * 8 + i] + tl[i]));
      }
    }
    // channels 0-2 to their own slots; a channel past them reuses slot 0 (stored already)
    const int slot_c = c < 3 ? c : 0;
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      const uint32_t lo = __byte_perm((uint32_t)xv[4 * k], (uint32_t)xv[4 * k + 1], 0x0040);
      const uint32_t hi = __byte_perm((uint32_t)xv[4 * k + 2], (uint32_t)xv[4 * k + 3], 0x0040);
      sOut[slot_c][threadIdx.x][k] = __byte_perm(lo, hi, 0x5410);
    }
    auto sample = [&](int q, int yy, int i) { return (int)__byte_perm(sOut[q][threadIdx.x][yy * 2 + (i >> 2)], 0u, 0x4440u + (i & 3)); };
    if (c >= 3) {  // a plain channel past the colour group: straight out
      for (int yy = ya; yy < yb; ++yy)
        for (int i = xa; i < xb; ++i) out(yy, i)[c] = (uint8_t)sample(0, yy, i);
    } else if (c == ngroup - 1) {  // channels 0 .. ngroup - 1 done: inverse colour map and store
      for (int yy = ya; yy < yb; ++yy)
        for (int i = xa; i < xb; ++i) {
          int ch[3];
#pragma unroll
          for (int q = 0; q < 3; ++q) ch[q] = q < ngroup ? sample(q, yy, i) : 0;
          if (ycbcr) {
            const int Y = ch[0], cb = 2 * ch[1] - 255, cr = 2 * ch[2] - 255;
            const int G = Y - ((cb + cr + 2) >> 2);
            ch[0] = clamp255(G + cr);
            ch[1] = clamp255(G);
            ch[2] = clamp255(G + cb);
          }
          uint8_t *p = out(yy, i);
#pragma unroll
          for (int q = 0; q < 3; ++q)
            if (q < ngroup) p[q] = (uint8_t)ch[q];
        }
    }
  }
}

// ---- scaled region decode: a rectangle of the image scaled by F = 2^lf ---------------------------------------------
// The rectangle [x, x + rw) x [y, y + rh) is given in the scaled image's coordinates; output pixel (Y, X) is the
// rounded box average of the source window at (F * Y, F * X), clipped at the right and bottom image edges, as in
// k_inverse_scaled.  Every window lies inside one block, so the blocks computed are those of the source rectangle
// [F x, min(F (x + rw), w)) x [F y, min(F (y + rh), h)), from the compact planes of k_dec_segtab_region_scaled.
//
//   k_inverse_region4_scaled  fast path (nch 1 / 3, w % 16 == 0, h % 8 == 0, cols % 16 == 0: every window whole):
//                             k_inverse_region4's tiles and inv4_compute's pooled output phase, clipped stores
//                             (Inv4StorePooledClip)
//   k_inverse_region_scaled   every other shape, force_generic and the mixed call: k_inverse_region's transform, then
//                             k_inverse_scaled's exact division per window

// Output row wy of a block pair's pooled lanes (see Inv4StorePooled), clipped to the rectangle.  The pair's
// 2 * (8 >> LF) * NCH bytes of a row are one run in the output at any byte alignment, of which the bytes [b0, b1)
// lie inside the rectangle: stored as Inv4StoreClip stores a full-size run.
template <int NCH, int LF>
struct Inv4StorePooledClip {
  uint8_t *row0;       // byte 0 of the pair's output row 0 (may lie outside the rectangle)
  long long row_bytes; // rw * NCH
  int y0, rh;          // output row 0 of the pair is row y0 of the rectangle
  int b0, b1;          // bytes of a run inside the rectangle
  __device__ __forceinline__ void operator()(int wy, const uint32_t (&p)[(8 >> LF) * NCH]) const {
    if (y0 + wy < 0 || y0 + wy >= rh) return;
    constexpr int K = (8 >> LF) * NCH, RB = 2 * K, NW = (RB + 3) / 4;  // bytes per block, per run, words of a run
    auto byte = [&](int b) -> uint32_t { return b < K ? (p[b] & 0xffu) : (p[b - K] >> 16); };
    uint32_t W[NW];
#pragma unroll
    for (int k = 0; k < NW; ++k) {
      W[k] = 0u;
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (4 * k + j < RB) W[k] |= byte(4 * k + j) << (8 * j);
    }
    const uintptr_t addr = reinterpret_cast<uintptr_t>(row0) + (uintptr_t)((long long)wy * row_bytes);
    const int a = (int)(addr & 3);
    uint8_t *base = reinterpret_cast<uint8_t *>(addr - (uintptr_t)a);
#pragma unroll
    for (int j = 0; j <= NW; ++j) {
      const int s = 4 * j - a;  // run byte at the output word's byte 0
      if (s >= b1 || s + 4 <= b0) continue;
      const uint32_t v = __funnelshift_rc(j > 0 ? W[j - 1] : 0u, j < NW ? W[j] : 0u, 8 * (4 - a));
      if (s >= b0 && s + 4 <= b1) {
        *reinterpret_cast<uint32_t *>(base + 4 * j) = v;
      } else {
#pragma unroll
        for (int t = 0; t < 4; ++t)
          if (s + t >= b0 && s + t < b1) base[4 * j + t] = (uint8_t)(v >> (8 * t));
      }
    }
  }
};

// grid (ceil(kr * span / TP), 1, n) with span = region_span_pairs(rw << LF, cols), block TP, dynamic smem as
// k_inverse4.  k_inverse_region4 on the source rectangle, with the output phase of k_inverse4_scaled.
template <int NCH, int TP, int LF>
__global__ void __launch_bounds__(TP, NCH == 1 ? 3 : 2)
    k_inverse_region4_scaled(const uint8_t *__restrict__ planes, const uint8_t *__restrict__ R, Geom g,
                             const InvTables *__restrict__ tabs, unsigned long long tab_stride,
                             const int32_t *__restrict__ origins, int rw, int rh, int kr, int span, uint8_t *__restrict__ pixels,
                             uint32_t one) {
  extern __shared__ __align__(128) uint8_t sPl[];
  constexpr int PITCH = 2 * TP, CPR = TP / 8, OB = 8 >> LF;  // OB: output pixels of a block per row
  static_assert(TP % 32 == 0 && TP == 8 * CPR, "a CTA is 8 groups of one thread per chunk of a tile row");
  uint8_t *sDq = sPl + NCH * 64 * PITCH;
  uint32_t *sTab = reinterpret_cast<uint32_t *>(sDq + kInvSlots * 256 * 2);
  const int item = blockIdx.z;
  int x, y;
  if (!region_origin_scaled(origins, item, g, LF, rw, rh, x, y)) return;  // (the whole CTA)
  const int t = threadIdx.x;
  const int sx = x << LF, sy = y << LF;  // (every window is whole: the source rectangle is (rw << LF) x (rh << LF))
  const int r0 = sy >> 3, r1 = (sy + (rh << LF) - 1) >> 3;
  const int u0 = (sx >> 3) & ~15, ul = sx >> 3, ur = (sx + (rw << LF) - 1) >> 3;
  const int f0 = blockIdx.x * TP, nact = min(TP, kr * span - f0);
  const uint8_t *ipl = planes + (size_t)item * kr * g.seg;
  const InvTables *T = reinterpret_cast<const InvTables *>(reinterpret_cast<const char *>(tabs) + (size_t)item * tab_stride);
  {
    const uint4 *tsrc = reinterpret_cast<const uint4 *>(T);
    for (int i = t; i < kInvTableBytes / 16; i += TP) cp_async16(sDq + 16 * i, tsrc + i);
    // a chunk = 8 pairs of one slot (span % 8 == 0), inside the image or wholly outside it (cols % 16 == 0)
    const int cq = t % CPR, rt = t / CPR, e = f0 + 8 * cq;
    const int s = e / span, u = u0 + 2 * (e - s * span);
    if (8 * cq < nact && u < g.cols) {
      const uint8_t *src = ipl + (size_t)s * g.seg + u + (size_t)rt * g.cols;
      uint8_t *dst = sPl + rt * PITCH + cq * 16;
      const size_t rstep = (size_t)8 * g.cols;
#pragma unroll 8
      for (int i = 0; i < NCH * 8; ++i) {
        cp_async16(dst + i * 8 * PITCH, src);
        src += rstep;
      }
    }
  }
  const int e = f0 + t, s = e / span;
  int u = u0 + 2 * (e - s * span);
  const bool active = t < nact && r0 + s <= r1 && u < g.cols && u + 1 >= ul && u <= ur;
  if (!active) u = u0;  // (corner loads inside the image)
  const int v = min(r0 + s, r1);
  uint32_t top[NCH], bot[NCH];
  inv4_corners<NCH>(R, item, g, v, u, top, bot);
  const int X0 = OB * u - x;  // rectangle column of the pair's first output pixel
  const Inv4StorePooledClip<NCH, LF> store{pixels + (size_t)item * rw * rh * NCH + ((long long)(OB * v - y) * rw + X0) * NCH,
                                           (long long)rw * NCH, OB * v - y, rh, max(0, -X0) * NCH, min(2 * OB, rw - X0) * NCH};
  const int pre = T->pre, tab_bias = T->bias;
  const bool overflow = T->overflow != 0;
  const bool ycbcr = T->ycbcr != 0;
  cp_async_wait_all();
  __syncthreads();
  inv4_compute<NCH, PITCH, Inv4StorePooledClip<NCH, LF>, LF>(sPl + 2 * t, sDq, sTab, pre, tab_bias, overflow, ycbcr, active, top,
                                                              bot, store, one);
}

// grid (ceil(kb / kTile), kr, n), block kTile (kb = ((rw << lf) + 15 - (1 << lf)) / 8 block columns): thread = block
// column (x << lf) / 8 + i of compact slot blockIdx.y.  k_inverse_region's transform and MIXED; the colour map is applied
// in place in shared memory, then every window of the thread's block inside the rectangle is averaged with one exact
// division per channel, as in k_inverse_scaled, and stored as bytes.
template <bool MIXED = false>
__global__ void __launch_bounds__(kTile)
    k_inverse_region_scaled(const uint8_t *__restrict__ planes, const uint8_t *__restrict__ R, Geom g,
                            const DecTables *__restrict__ tabs, unsigned long long tab_stride, const int32_t *__restrict__ origins,
                            int rw, int rh, int kr, int lf, uint8_t *__restrict__ pixels, MixedDims md = {}) {
  __shared__ int16_t sUn[256];
  __shared__ uint8_t sShift[2][64];
  __shared__ uint32_t sOut[3][kTile][17];  // channels 0-2 of a thread's block (the colour map needs all three)
  const int item = blockIdx.z, slot = blockIdx.y;
  Geom gi = g;  // the image's geometry
  if (MIXED && !image_geom(md, item, gi)) return;
  int x, y;
  if (!region_origin_scaled(origins, item, gi, lf, rw, rh, x, y)) return;  // (the whole CTA)
  const int f = 1 << lf;
  const int sx = x << lf, sy = y << lf, sx1 = min((x + rw) << lf, gi.w), sy1 = min((y + rh) << lf, gi.h);
  const int v = (sy >> 3) + slot;
  if (v > (sy1 - 1) >> 3) return;  // a repeated slot
  const DecTables *T = reinterpret_cast<const DecTables *>(reinterpret_cast<const char *>(tabs) + (size_t)item * tab_stride);
  for (int i = threadIdx.x; i < 256; i += blockDim.x) sUn[i] = T->full_unmap[i];
  for (int i = threadIdx.x; i < 128; i += blockDim.x) sShift[i >> 6][i & 63] = T->shift[i >> 6][i & 63];
  const int nch = g.nch;
  const bool ycbcr = T->ycbcr != 0 && nch >= 3;
  __syncthreads();
  const int u = (sx >> 3) + blockIdx.x * kTile + threadIdx.x;
  if (u > (sx1 - 1) >> 3) return;
  const uint8_t *seg = MIXED ? planes + (size_t)item * kr * g.seg + (size_t)slot * gi.seg : planes + ((size_t)item * kr + slot) * g.seg;
  uint8_t *img = pixels + (size_t)item * rw * rh * nch;
  // windows of the block inside the rectangle: [wya, wyb) x [wxa, wxb); window (wy, wx) is output pixel (oy0 + wy, ox0 + wx)
  const int bh = min(8, gi.h - 8 * v), bw = min(8, gi.w - 8 * u);
  const int oy0 = (8 * v) >> lf, ox0 = (8 * u) >> lf;
  const int wya = max(0, y - oy0), wyb = min((bh + f - 1) >> lf, y + rh - oy0);
  const int wxa = max(0, x - ox0), wxb = min((bw + f - 1) >> lf, x + rw - ox0);
  // rounded average of window (wy, wx) of a block's 64 bytes (pixel 8 * row + column)
  auto pool = [&](const uint8_t *px, int wy, int wx) -> uint8_t {
    const int ny = min(f, bh - wy * f), nx = min(f, bw - wx * f), n = nx * ny, p0 = wy * f * 8 + wx * f;
    int S = 0;
    for (int yy = 0; yy < ny; ++yy)
      for (int xx = 0; xx < nx; ++xx) S += px[p0 + yy * 8 + xx];
    return (uint8_t)((S + (n >> 1)) / n);
  };
  auto out = [&](int wy, int wx) { return img + ((size_t)(oy0 + wy - y) * rw + (ox0 + wx - x)) * nch; };
  const int ngroup = min(nch, 3);
#pragma unroll 1
  for (int c = 0; c < nch; ++c) {
    int xv[64];
    const uint8_t *src = seg + (size_t)c * gi.cols * 64 + u;
    const uint8_t *sh = sShift[(ycbcr && (c == 1 || c == 2)) ? 1 : 0];
#pragma unroll
    for (int j = 0; j < 64; ++j) xv[j] = (int)(short)(sUn[__ldg(src + (size_t)scan_pos(j) * gi.cols)] * (1 << sh[j]));
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      wht8(xv[r * 8 + 0], xv[r * 8 + 1], xv[r * 8 + 2], xv[r * 8 + 3], xv[r * 8 + 4], xv[r * 8 + 5], xv[r * 8 + 6], xv[r * 8 + 7]);
#pragma unroll
      for (int i = 0; i < 8; ++i) xv[r * 8 + i] >>= 3;
    }
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      wht8(xv[q], xv[8 + q], xv[16 + q], xv[24 + q], xv[32 + q], xv[40 + q], xv[48 + q], xv[56 + q]);
#pragma unroll
      for (int i = 0; i < 8; ++i) xv[i * 8 + q] >>= 3;
    }
    {
      const LowCorners k =
          load_corners(MIXED ? R + (size_t)item * nch * g.rows * g.cols + (size_t)c * gi.rows * gi.cols : R + ((size_t)item * nch + c) * g.rows * g.cols,
                       gi, u, v);
      int lf9[9], rt9[9];
      nine(k.x11, k.x21, lf9);
      nine(k.x12, k.x22, rt9);
#pragma unroll
      for (int yy = 0; yy < 8; ++yy) {
        int tl[9];
        nine(lf9[yy], rt9[yy], tl);
#pragma unroll
        for (int i = 0; i < 8; ++i) xv[yy * 8 + i] = clamp255((int)(short)(xv[yy * 8 + i] + tl[i]));
      }
    }
    // channels 0-2 to their own slots; a channel past them reuses slot 0 (stored already)
    const int slot_c = c < 3 ? c : 0;
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      const uint32_t lo = __byte_perm((uint32_t)xv[4 * k], (uint32_t)xv[4 * k + 1], 0x0040);
      const uint32_t hi = __byte_perm((uint32_t)xv[4 * k + 2], (uint32_t)xv[4 * k + 3], 0x0040);
      sOut[slot_c][threadIdx.x][k] = __byte_perm(lo, hi, 0x5410);
    }
    uint8_t *px[3];  // pixel p = 8 * row + column of slot q: px[q][p]
#pragma unroll
    for (int q = 0; q < 3; ++q) px[q] = reinterpret_cast<uint8_t *>(&sOut[q][threadIdx.x][0]);
    if (c >= 3) {  // a plain channel past the colour group: straight out
      for (int wy = wya; wy < wyb; ++wy)
        for (int wx = wxa; wx < wxb; ++wx) out(wy, wx)[c] = pool(px[0], wy, wx);
    } else if (c == ngroup - 1) {  // channels 0 .. ngroup - 1 done: inverse colour map in place, then the averages
      if (ycbcr) {
#pragma unroll 4
        for (int p = 0; p < 64; ++p) {
          const int Y = px[0][p], cb = 2 * px[1][p] - 255, cr = 2 * px[2][p] - 255;
          const int G = Y - ((cb + cr + 2) >> 2);
          px[0][p] = (uint8_t)clamp255(G + cr);
          px[1][p] = (uint8_t)clamp255(G);
          px[2][p] = (uint8_t)clamp255(G + cb);
        }
      }
      for (int wy = wya; wy < wyb; ++wy)
        for (int wx = wxa; wx < wxb; ++wx) {
          uint8_t *o = out(wy, wx);
          for (int q = 0; q < ngroup; ++q) o[q] = pool(px[q], wy, wx);
        }
    }
  }
}

}  // namespace himgcu

#endif  // HIMG_B200_XFORM_REGION_CUH_
