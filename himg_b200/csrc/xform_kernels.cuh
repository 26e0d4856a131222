// Transform-side kernels: colour mapping, low-res (DC) image + DPCM, forward / inverse 8x8 WHT with
// shift quantisation and 8-bit mapping.  All integer, no tensor cores (the work is +-1 add/sub and
// HBM bound); thread = one 8x8 pixel block with the butterflies fully unrolled in registers.
#ifndef HIMG_B200_XFORM_KERNELS_CUH_
#define HIMG_B200_XFORM_KERNELS_CUH_

#include "common.cuh"

namespace himgcu {

constexpr int kTile = 128;  // blocks (threads) per CTA along x

// ---------------------------------------------------------------------------------------------
// Pixel row access.  A "row" is the 8 horizontally adjacent pixels of one block row; the fast
// path reads them as 2*NCH aligned 32-bit words straight from HBM (a warp covers 32*8*NCH
// contiguous bytes), the slow path handles pixel_stride != NCH, unaligned rows and the right
// image edge, replicating the last valid pixel like ExtractChannelBlock (encoder.cpp:26-52).
// ---------------------------------------------------------------------------------------------
template <int NCH>
struct Row8 {
  uint32_t w[2 * NCH];
  __device__ __forceinline__ int byte(int k) const { return (int)__byte_perm(w[k >> 2], 0u, 0x4440u + (k & 3)); }
  __device__ __forceinline__ int px(int i, int c) const { return byte(i * NCH + c); }
};

template <int NCH>
__device__ __forceinline__ void load_row8(Row8<NCH> &r, const uint8_t *__restrict__ img, const Geom &g,
                                          int y, int u, bool fast) {
  const uint8_t *p = img + ((size_t)y * g.w + (size_t)u * 8) * g.pstride;
  if (fast) {
    const uint2 *q = reinterpret_cast<const uint2 *>(p);
#pragma unroll
    for (int k = 0; k < NCH; ++k) {
      const uint2 t = __ldg(q + k);
      r.w[2 * k] = t.x;
      r.w[2 * k + 1] = t.y;
    }
  } else {
#pragma unroll
    for (int k = 0; k < 2 * NCH; ++k) r.w[k] = 0;
    const int xmax = g.w - 1 - u * 8;  // last valid pixel inside this block
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int xi = i < xmax ? i : xmax;
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        const uint32_t b = p[(size_t)xi * g.pstride + c];
        const int k = i * NCH + c;
        r.w[k >> 2] |= b << (8 * (k & 3));
      }
    }
  }
}

template <int NCH>
__device__ __forceinline__ bool row_fast_ok(const uint8_t *img, const Geom &g, int u) {
  return g.pstride == NCH && (u * 8 + 8 <= g.w) && (((size_t)g.w * NCH) & 7) == 0 &&
         ((reinterpret_cast<uintptr_t>(img)) & 7) == 0;
}

// Colour mapping of one pixel's channel c (ycbcr.cpp:24-52).
template <int NCH, bool YCBCR>
__device__ __forceinline__ int colour_fwd(const Row8<NCH> &r, int i, int c) {
  if (YCBCR && NCH >= 3 && c < 3) {
    const int R = r.px(i, 0), G = r.px(i, 1), B = r.px(i, 2);
    if (c == 0) return (R + 2 * G + B + 2) >> 2;
    if (c == 1) return (B - G + 256) >> 1;
    return (R - G + 256) >> 1;
  }
  return r.px(i, c);
}

// ---------------------------------------------------------------------------------------------
// K-avg: per block corner (u,v), mean of the colour-mapped pixels in the 8x8 window centred on
// the block's top-left corner, clipped to the image (downsampled.cpp:75-94).
// grid (ceil(cols/kTile), rows, n), block kTile.  avg: [n][nch][rows][cols].
// ---------------------------------------------------------------------------------------------
// Channel groups: an image of more than four channels (the reference passes any number through,
// ycbcr.cpp:24-52, encoder.cpp:69) is handled as its first three channels (colour mapped or not) plus one
// launch per further channel.  `pixels` then points at the group's first channel (g.pstride = all channels)
// and cbase / ctotal place the group's planes among the image's: [n][ctotal][rows][cols].
// MIXED (encode of a mixed-geometry batch): g is the bounding geometry, which sets the grid and the slot of
// ctotal * rows * cols bytes per image; image z starts at pixels + px_off[z] and is averaged with its own geometry
// from `md`, its planes [ctotal][rows][cols] of that geometry at the start of its slot.  Blocks outside it, and
// images with dims out of bounds, are idle.
template <int NCH, bool YCBCR, bool MIXED = false>
__global__ void __launch_bounds__(kTile) k_lowres_avg(const uint8_t *__restrict__ pixels, Geom g,
                                                      uint8_t *__restrict__ avg, int cbase, int ctotal, MixedDims md = {},
                                                      const unsigned long long *__restrict__ px_off = nullptr) {
  __shared__ int sB[NCH][kTile + 1];
  const int v = blockIdx.y, t0 = blockIdx.x * kTile, u = t0 + threadIdx.x;
  const Geom gb = g;  // bounding geometry (slot strides)
  if (MIXED && (!image_geom(md, blockIdx.z, g) || t0 >= g.cols || v >= g.rows)) return;  // (uniform per CTA)
  const uint8_t *img = MIXED ? pixels + px_off[blockIdx.z] : pixels + (size_t)blockIdx.z * g.img_bytes;
  const int y0 = max(0, 8 * v - 3), y1 = min(g.h - 1, 8 * v + 4);
  int A[NCH], B[NCH];
#pragma unroll
  for (int c = 0; c < NCH; ++c) A[c] = B[c] = 0;
  if (u < g.cols) {
    const bool fast = row_fast_ok<NCH>(img, g, u);
    const int nvalid = min(8, g.w - 8 * u);
    for (int y = y0; y <= y1; ++y) {
      Row8<NCH> r;
      load_row8<NCH>(r, img, g, y, u, fast);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        if (i < nvalid) {
#pragma unroll
          for (int c = 0; c < NCH; ++c) {
            const int val = colour_fwd<NCH, YCBCR>(r, i, c);
            if (i < 5) A[c] += val;
            else B[c] += val;
          }
        }
      }
    }
  }
#pragma unroll
  for (int c = 0; c < NCH; ++c) sB[c][threadIdx.x + 1] = B[c];
  if (threadIdx.x == 0) {
    // right-hand three columns of the block left of this tile
    int Bl[NCH];
#pragma unroll
    for (int c = 0; c < NCH; ++c) Bl[c] = 0;
    if (t0 > 0) {
      Row8<NCH> r;
      const bool fast = row_fast_ok<NCH>(img, g, t0 - 1);
      for (int y = y0; y <= y1; ++y) {
        load_row8<NCH>(r, img, g, y, t0 - 1, fast);
#pragma unroll
        for (int i = 5; i < 8; ++i)
#pragma unroll
          for (int c = 0; c < NCH; ++c) Bl[c] += colour_fwd<NCH, YCBCR>(r, i, c);
      }
    }
#pragma unroll
    for (int c = 0; c < NCH; ++c) sB[c][0] = Bl[c];
  }
  __syncthreads();
  if (u < g.cols) {
    const int nx = min(g.w - 1, 8 * u + 4) - max(0, 8 * u - 3) + 1;
    const int cnt = nx * (y1 - y0 + 1);
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      const int s = A[c] + sB[c][threadIdx.x];
      if (MIXED)
        avg[(size_t)blockIdx.z * ctotal * gb.rows * gb.cols + ((size_t)(cbase + c) * g.rows + v) * g.cols + u] =
            (uint8_t)((s + (cnt >> 1)) / cnt);
      else
        avg[(((size_t)blockIdx.z * ctotal + cbase + c) * g.rows + v) * g.cols + u] = (uint8_t)((s + (cnt >> 1)) / cnt);
    }
  }
}

// 1/16-pixel phase compensation (downsampled.cpp:96-113): L = blend(blend(row v-1), blend(row v)) with
// blend(row r) = (a[r][u-1] + 15 a[r][u] + 8) >> 4, edges clamped.  A thread owns column u of
// kCompRows consecutive rows and computes every row blend once (the lower blend of row v is the upper
// blend of row v+1); 32-bit indices only (a 64-bit division per sample was most of the first version).
// grid (planes, ceil(rows / kCompRows)), any block size (threads stride over the columns).
// MIXED: rows x cols is the bounding geometry and plane p is channel p % md.nch of image p / md.nch, laid out with
// that image's rows and cols inside its slot of md.nch * rows * cols bytes (as k_lowres_avg<.., true> writes it).
constexpr int kCompRows = 4;
template <bool MIXED = false>
__global__ void k_lowres_comp(const uint8_t *__restrict__ avg, int planes, int rows, int cols,
                              uint8_t *__restrict__ L, MixedDims md = {}) {
  size_t base = (size_t)blockIdx.x * rows * cols;
  if (MIXED) {
    const int img = blockIdx.x / md.nch, c = blockIdx.x - img * md.nch;
    Geom gi;
    if (!image_geom(md, img, gi) || (int)blockIdx.y * kCompRows >= gi.rows) return;
    base = (size_t)img * md.nch * rows * cols + (size_t)c * gi.rows * gi.cols;
    rows = gi.rows;
    cols = gi.cols;
  }
  const uint8_t *a = avg + base;
  uint8_t *o = L + base;
  const int v0 = blockIdx.y * kCompRows;
  for (int u = threadIdx.x; u < cols; u += blockDim.x) {
    const int up = max(u - 1, 0);
    const int rp = max(v0 - 1, 0);
    int prev = (a[rp * cols + up] + 15 * a[rp * cols + u] + 8) >> 4;
#pragma unroll
    for (int k = 0; k < kCompRows; ++k) {
      const int v = v0 + k;
      if (v < rows) {
        const int cur = (a[v * cols + up] + 15 * a[v * cols + u] + 8) >> 4;
        o[v * cols + u] = (uint8_t)((prev + 15 * cur + 8) >> 4);
        prev = cur;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Low-res DPCM (downsampled.cpp:33-60, :177-382).  Half a warp = one 16x16 macroblock: predictor
// selection by parallel SSE, then the reconstruction-dependent DPCM as a 31-step anti-diagonal
// wavefront (lane = column).  Nothing crosses a macroblock edge, so macroblocks are independent.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ int lres_predict(int s1, int s2, int s3, int p) {
  switch (p) {
    case 1: return s2;
    case 2: return s3;
    case 3: return (s2 + s3 + 1) >> 1;
    case 4: return clamp255(s2 + s3 - s1);
    default: return clamp255((3 * (s2 + s3) - 2 * s1 + 2) >> 2);
  }
}

struct LowResTables {
  uint8_t map_lut[256];    // |delta| -> magnitude code (encoder only)
  int16_t unmap[256];      // code byte -> value (Mapper::UnmapFrom8Bit)
};
// The DPCM kernel reads its tables through the read-only path: `unmap` may be per image
// (decoder: tables travel in-band) with `unmap_stride` bytes between images, or shared (stride 0).

constexpr int kLresWarps = 4;

// MIXED (mixed-geometry batch, encode or decode): g is the bounding geometry, which sets the grid and the slot strides
// (lres_stride and nch * rows * cols bytes per image); image img's macroblocks and its layout inside the slots are
// those of its own geometry from `md`.  Macroblocks outside it, and images with dims out of bounds, are idle.
template <bool ENCODE, bool MIXED = false>
__global__ void __launch_bounds__(kLresWarps * 32)
    k_lres_dpcm(const uint8_t *__restrict__ Lin,   // ENCODE: L [n][nch][rows][cols]; else unused
                uint8_t *__restrict__ lres,        // ENCODE: out; DECODE: in  ([n][lres_stride])
                uint8_t *__restrict__ Rout,        // DECODE: R [n][nch][rows][cols]
                Geom g, int n, const uint8_t *__restrict__ map_lut, const int16_t *__restrict__ unmap,
                unsigned long long unmap_stride, MixedDims md = {}) {
  __shared__ uint8_t sL[kLresWarps * 2][16][16];
  __shared__ uint8_t sR[kLresWarps * 2][16][17];
  // The codes of a macroblock are contiguous in memory but the wavefront touches them along
  // diagonals: one byte per lane and step would be one 32-byte L2 transaction per byte.  They pass
  // through shared memory and move in rows of consecutive bytes instead (as do the decoded samples).
  __shared__ uint8_t sC[kLresWarps * 2][256];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, half = lane >> 4, hl = lane & 15;
  const long long nmb = (long long)n * g.nch * g.mrows * g.mcols;
  const long long mb = ((long long)blockIdx.x * kLresWarps + wid) * 2 + half;
  bool active = mb < nmb;
  const int slot = wid * 2 + half;
  int img = 0, c = 0, mv = 0, mu = 0;
  if (active) {
    long long t = mb;
    mu = (int)(t % g.mcols);
    t /= g.mcols;
    mv = (int)(t % g.mrows);
    t /= g.mrows;
    c = (int)(t % g.nch);
    img = (int)(t / g.nch);
  }
  Geom gi = g;  // image img's geometry
  if (MIXED) {
    active = active && image_geom(md, img, gi) && mv < gi.mrows && mu < gi.mcols;
    if (!active) mv = mu = 0;
  }
  const int bh = min(16, gi.rows - 16 * mv), bw = min(16, gi.cols - 16 * mu);
  const int16_t *un = reinterpret_cast<const int16_t *>(reinterpret_cast<const char *>(unmap) + (size_t)img * unmap_stride);
  const size_t plane = MIXED ? (size_t)img * g.nch * g.rows * g.cols + (size_t)c * gi.rows * gi.cols
                             : ((size_t)img * g.nch + c) * g.rows * g.cols;
  uint8_t *chan = lres + (size_t)img * g.lres_stride + (size_t)c * gi.lres_ch;
  uint8_t *selp = chan + mv * gi.mcols + mu;
  uint8_t *dp = chan + gi.mrows * gi.mcols + (size_t)mv * 16 * gi.cols + (size_t)mu * 16 * bh;

  int p = 0;
  if (ENCODE) {
    // stage the macroblock (row hl) and pick the predictor
    if (active && hl < bw)  // lane = column: every load instruction reads one row of consecutive bytes
      for (int dv = 0; dv < bh; ++dv) sL[slot][dv][hl] = __ldg(Lin + plane + (size_t)(16 * mv + dv) * gi.cols + 16 * mu + hl);
    __syncwarp();
    int err[5] = {0, 0, 0, 0, 0};
    if (active && hl < bh) {
      const int dv = hl;
      for (int du = 0; du < bw; ++du) {
        int s1, s2, s3;
        if (du > 0 && dv > 0) {
          s1 = sL[slot][dv - 1][du - 1];
          s2 = sL[slot][dv - 1][du];
          s3 = sL[slot][dv][du - 1];
        } else if (du > 0) {
          s1 = s2 = s3 = sL[slot][dv][du - 1];
        } else if (dv > 0) {
          s1 = s2 = s3 = sL[slot][dv - 1][du];
        } else {
          s1 = s2 = s3 = 128;
        }
        const int actual = sL[slot][dv][du];
#pragma unroll
        for (int q = 0; q < 5; ++q) {
          const int d = actual - lres_predict(s1, s2, s3, q);
          err[q] += d * d;
        }
      }
    }
#pragma unroll
    for (int q = 0; q < 5; ++q)
#pragma unroll
      for (int d = 8; d >= 1; d >>= 1) err[q] += __shfl_xor_sync(0xffffffffu, err[q], d);
    int best = 0;
#pragma unroll
    for (int q = 1; q < 5; ++q)
      if (err[q] < err[best]) best = q;
    const int sel = (best - 2) & 0xff;  // EncodePredictor (downsampled.cpp:33-35)
    if (active && hl == 0) *selp = (uint8_t)sel;
    p = sel + 2;  // DecodePredictor widens first: 254/255 -> 256/257 -> default formula
  } else {
    if (active) {
      p = (int)(*selp) + 2;
      for (int i = hl; i < bh * bw; i += 16) sC[slot][i] = dp[i];
    }
    __syncwarp();
  }

  // wavefront: lane hl owns column du = hl; at step s it handles row dv = s - du
  for (int s = 0; s < 31; ++s) {
    const int du = hl, dv = s - du;
    if (active && dv >= 0 && dv < bh && du < bw) {
      int s1, s2, s3;
      if (du > 0 && dv > 0) {
        s1 = sR[slot][dv - 1][du - 1];
        s2 = sR[slot][dv - 1][du];
        s3 = sR[slot][dv][du - 1];
      } else if (du > 0) {
        s1 = s2 = s3 = sR[slot][dv][du - 1];
      } else if (dv > 0) {
        s1 = s2 = s3 = sR[slot][dv - 1][du];
      } else {
        s1 = s2 = s3 = 128;
      }
      const int pr = lres_predict(s1, s2, s3, p);
      int code;
      if (ENCODE) {
        const int d = (int)sL[slot][dv][du] - pr;
        const int m = __ldg(map_lut + (d < 0 ? -d : d));
        code = d >= 0 ? m : ((256 - m) & 0xff);
        sC[slot][dv * bw + du] = (uint8_t)code;
      } else {
        code = sC[slot][dv * bw + du];
      }
      const int rec = clamp255((int)(short)(pr + __ldg(un + code)));
      sR[slot][dv][du] = (uint8_t)rec;
    }
    __syncwarp();
  }
  if (active) {
    if (ENCODE) {
      for (int i = hl; i < bh * bw; i += 16) dp[i] = sC[slot][i];
    } else if (hl < bw) {
      for (int dv = 0; dv < bh; ++dv) Rout[plane + (size_t)(16 * mv + dv) * gi.cols + 16 * mu + hl] = sR[slot][dv][hl];
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Bilinear-by-midpoints 8x8 patch of the low-res image (downsampled.cpp:116-169): rows first get
// their left/right end points from the vertical interpolation, then each row is interpolated.
// ---------------------------------------------------------------------------------------------
struct LowCorners {
  int x11, x12, x21, x22;
};
__device__ __forceinline__ LowCorners load_corners(const uint8_t *__restrict__ X, const Geom &g, int u, int v) {
  const int v2 = min(v + 1, g.rows - 1), u2 = min(u + 1, g.cols - 1);
  LowCorners k;
  k.x11 = __ldg(X + v * g.cols + u);
  k.x12 = __ldg(X + v * g.cols + u2);
  k.x21 = __ldg(X + v2 * g.cols + u);
  k.x22 = __ldg(X + v2 * g.cols + u2);
  return k;
}

// ---------------------------------------------------------------------------------------------
// K-fwd (the roofline kernel): colour map + low-res subtract + rows/cols WHT + shift quantise +
// 8-bit map + coefficient-planar scatter (encoder.cpp:275-328, hadamard.cpp:78-88,
// quantize.cpp:127-151, mapper.cpp:159-182).  grid (ceil(cols/kTile), rows, n), block kTile.
// Algorithmic traffic: nch bytes read + nch bytes written per pixel.
// ---------------------------------------------------------------------------------------------
// MIXED (encode of a mixed-geometry batch): g is the bounding geometry (grid; slots of planes_bytes in `planes` and
// of ctotal * rows * cols in L); image z starts at pixels + px_off[z], and its blocks, edges, low-res planes and
// segments (gi.seg bytes each, from the start of its slot) are those of its own geometry from `md`.
template <int NCH, bool YCBCR, bool MIXED = false>
__global__ void __launch_bounds__(kTile)
    k_forward(const uint8_t *__restrict__ pixels, const uint8_t *__restrict__ L, Geom g,
              const __grid_constant__ QuantParams qp, const uint8_t *__restrict__ map_lut,
              uint8_t *__restrict__ planes, int cbase, int ctotal, MixedDims md = {},
              const unsigned long long *__restrict__ px_off = nullptr) {
  __shared__ uint8_t sLut[7616];
  {
    const uint4 *src = reinterpret_cast<const uint4 *>(map_lut);
    uint4 *dst = reinterpret_cast<uint4 *>(sLut);
    for (int i = threadIdx.x; i < 7616 / 16; i += blockDim.x) dst[i] = __ldg(src + i);
  }
  __syncthreads();
  const int v = blockIdx.y, u = blockIdx.x * kTile + threadIdx.x;
  const Geom gb = g;  // bounding geometry (slot strides)
  const uint8_t *img;
  if (MIXED) {
    if (!image_geom(md, blockIdx.z, g) || v >= g.rows) return;
    img = pixels + px_off[blockIdx.z];
  }
  if (u >= g.cols) return;
  if (!MIXED) img = pixels + (size_t)blockIdx.z * g.img_bytes;
  const bool fast = row_fast_ok<NCH>(img, g, u);
  const int bh = min(8, g.h - 8 * v);
  uint8_t *seg = planes + (size_t)blockIdx.z * gb.planes_bytes + (size_t)v * g.seg;

#pragma unroll 1
  for (int c = 0; c < NCH; ++c) {
    int x[64];
    int last = 0;
    // ---- extract (with the reference's edge replication) + colour map
#pragma unroll
    for (int y = 0; y < 8; ++y) {
      if (y < bh) {
        Row8<NCH> r;
        load_row8<NCH>(r, img, g, 8 * v + y, u, fast);
        if (c == 0) {
#pragma unroll
          for (int i = 0; i < 8; ++i) x[y * 8 + i] = colour_fwd<NCH, YCBCR>(r, i, 0);
        } else if (c == 1) {
#pragma unroll
          for (int i = 0; i < 8; ++i) x[y * 8 + i] = colour_fwd<NCH, YCBCR>(r, i, NCH > 1 ? 1 : 0);
        } else if (c == 2) {
#pragma unroll
          for (int i = 0; i < 8; ++i) x[y * 8 + i] = colour_fwd<NCH, YCBCR>(r, i, NCH > 2 ? 2 : 0);
        } else {
#pragma unroll
          for (int i = 0; i < 8; ++i) x[y * 8 + i] = colour_fwd<NCH, YCBCR>(r, i, NCH > 3 ? 3 : 0);
        }
        last = x[y * 8 + 7];
      } else {
        // rows below the image: the single last value written (bottom-right valid pixel)
#pragma unroll
        for (int i = 0; i < 8; ++i) x[y * 8 + i] = last;
      }
    }
    // ---- subtract the interpolated low-res patch (un-quantised L: SURVEY A.4-5)
    {
      const uint8_t *Lp = MIXED ? L + (size_t)blockIdx.z * ctotal * gb.rows * gb.cols + (size_t)(cbase + c) * g.rows * g.cols
                                : L + ((size_t)blockIdx.z * ctotal + cbase + c) * g.rows * g.cols;
      const LowCorners k = load_corners(Lp, g, u, v);
      int lf[9], rt[9];
      nine(k.x11, k.x21, lf);
      nine(k.x12, k.x22, rt);
#pragma unroll
      for (int y = 0; y < 8; ++y) {
        int t[9];
        nine(lf[y], rt[y], t);
#pragma unroll
        for (int i = 0; i < 8; ++i) x[y * 8 + i] -= t[i];
      }
    }
    // ---- 2-D WHT, rows then columns, unscaled (|T| <= 16320)
#pragma unroll
    for (int r = 0; r < 8; ++r)
      wht8(x[r * 8 + 0], x[r * 8 + 1], x[r * 8 + 2], x[r * 8 + 3], x[r * 8 + 4], x[r * 8 + 5], x[r * 8 + 6], x[r * 8 + 7]);
#pragma unroll
    for (int q = 0; q < 8; ++q)
      wht8(x[q], x[8 + q], x[16 + q], x[24 + q], x[32 + q], x[40 + q], x[48 + q], x[56 + q]);
    // ---- sign-magnitude rounding shift, map to 8 bit, scatter in scan order
    uint8_t *dst = seg + (size_t)(cbase + c) * g.cols * 64 + u;
    const bool chroma = YCBCR && NCH >= 3 && (c == 1 || c == 2);
    if (chroma) {
#pragma unroll
      for (int j = 0; j < 64; ++j) {
        const int t = x[j], a = t < 0 ? -t : t;
        const int m = min((a + qp.round[1][j]) >> qp.shift[1][j], 7608);
        const int code = sLut[m];
        dst[(size_t)scan_pos(j) * g.cols] = (uint8_t)(t < 0 ? -code : code);
      }
    } else {
#pragma unroll
      for (int j = 0; j < 64; ++j) {
        const int t = x[j], a = t < 0 ? -t : t;
        const int m = min((a + qp.round[0][j]) >> qp.shift[0][j], 7608);
        const int code = sLut[m];
        dst[(size_t)scan_pos(j) * g.cols] = (uint8_t)(t < 0 ? -code : code);
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// K-inv: gather + dequantise + inverse WHT (floor >>3 after each pass) + low-res add + clamp +
// inverse colour map + cropped store (decoder.cpp:366-423, quantize.cpp:153-165,
// hadamard.cpp:90-103, ycbcr.cpp:54-82).  Same grid as K-fwd; same algorithmic traffic.
// Width % 8 != 0 is undefined in the reference; here the block is cropped.
// ---------------------------------------------------------------------------------------------
// MIXED (whole-image decode of a mixed-geometry batch): g is the bounding geometry (grid; slots of planes_bytes in
// `planes` and of ctotal * rows * cols in R); image z is written at pixels + px_off[z], and its blocks, segments,
// low-res planes and edges are those of its own geometry from `md`.  An image with dims out of bounds is not written.
template <int NCH, bool MIXED = false>
__global__ void __launch_bounds__(kTile)
    k_inverse(const uint8_t *__restrict__ planes, const uint8_t *__restrict__ R, Geom g,
              const DecTables *__restrict__ tabs, unsigned long long tab_stride,
              uint8_t *__restrict__ pixels, int cbase, int ctotal, MixedDims md = {},
              const unsigned long long *__restrict__ px_off = nullptr) {
  __shared__ int16_t sUn[256];
  __shared__ uint8_t sShift[2][64];
  __shared__ uint32_t sOut[NCH][kTile][17];  // per channel: 64 result bytes per thread (+1 pad)
  const Geom gb = g;  // bounding geometry (slot strides)
  if (MIXED && (!image_geom(md, blockIdx.z, g) || (int)blockIdx.y >= g.rows || (int)blockIdx.x * kTile >= g.cols)) return;
  const DecTables *T = reinterpret_cast<const DecTables *>(reinterpret_cast<const char *>(tabs) + (size_t)blockIdx.z * tab_stride);
  for (int i = threadIdx.x; i < 256; i += blockDim.x) sUn[i] = T->full_unmap[i];
  for (int i = threadIdx.x; i < 128; i += blockDim.x) sShift[i >> 6][i & 63] = T->shift[i >> 6][i & 63];
  const bool YCBCR = T->ycbcr != 0 && cbase == 0;  // (only the first three channels of an image are colour mapped)
  __syncthreads();
  const int v = blockIdx.y, u = blockIdx.x * kTile + threadIdx.x;
  if (u >= g.cols) return;
  const int bh = min(8, g.h - 8 * v), bw = min(8, g.w - 8 * u);
  const uint8_t *seg = planes + (size_t)blockIdx.z * gb.planes_bytes + (size_t)v * g.seg;
  uint8_t *img = MIXED ? pixels + px_off[blockIdx.z] : pixels + (size_t)blockIdx.z * g.out_img_bytes;

#pragma unroll 1
  for (int c = 0; c < NCH; ++c) {
    int x[64];
    const uint8_t *src = seg + (size_t)(cbase + c) * g.cols * 64 + u;
    const uint8_t *sh = sShift[(YCBCR && NCH >= 3 && (c == 1 || c == 2)) ? 1 : 0];
#pragma unroll
    for (int j = 0; j < 64; ++j) {
      const int code = __ldg(src + (size_t)scan_pos(j) * g.cols);
      const int val = sUn[code];
      // (int16)(Unmap << shift): the narrowing only matters for hostile streams
      x[j] = (int)(short)(val * (1 << sh[j]));
    }
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      wht8(x[r * 8 + 0], x[r * 8 + 1], x[r * 8 + 2], x[r * 8 + 3], x[r * 8 + 4], x[r * 8 + 5], x[r * 8 + 6], x[r * 8 + 7]);
#pragma unroll
      for (int i = 0; i < 8; ++i) x[r * 8 + i] >>= 3;
    }
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      wht8(x[q], x[8 + q], x[16 + q], x[24 + q], x[32 + q], x[40 + q], x[48 + q], x[56 + q]);
#pragma unroll
      for (int i = 0; i < 8; ++i) x[i * 8 + q] >>= 3;
    }
    {
      const uint8_t *Rp = MIXED ? R + (size_t)blockIdx.z * ctotal * gb.rows * gb.cols + (size_t)(cbase + c) * g.rows * g.cols
                                : R + ((size_t)blockIdx.z * ctotal + cbase + c) * g.rows * g.cols;
      const LowCorners k = load_corners(Rp, g, u, v);
      int lf[9], rt[9];
      nine(k.x11, k.x21, lf);
      nine(k.x12, k.x22, rt);
#pragma unroll
      for (int y = 0; y < 8; ++y) {
        int t[9];
        nine(lf[y], rt[y], t);
#pragma unroll
        for (int i = 0; i < 8; ++i) x[y * 8 + i] = clamp255((int)(short)(x[y * 8 + i] + t[i]));
      }
    }
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      const uint32_t lo = __byte_perm((uint32_t)x[4 * k], (uint32_t)x[4 * k + 1], 0x0040);
      const uint32_t hi = __byte_perm((uint32_t)x[4 * k + 2], (uint32_t)x[4 * k + 3], 0x0040);
      sOut[c][threadIdx.x][k] = __byte_perm(lo, hi, 0x5410);
    }
  }

  // ---- inverse colour map + interleave + store
  const bool aligned = ctotal == NCH && bw == 8 && (((size_t)g.w * NCH) & 7) == 0 && ((reinterpret_cast<uintptr_t>(img)) & 7) == 0;
#pragma unroll
  for (int y = 0; y < 8; ++y) {
    if (y < bh) {
      uint32_t ow[2 * NCH];
#pragma unroll
      for (int k = 0; k < 2 * NCH; ++k) ow[k] = 0;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        int ch[NCH];
#pragma unroll
        for (int c = 0; c < NCH; ++c) ch[c] = (int)__byte_perm(sOut[c][threadIdx.x][y * 2 + (i >> 2)], 0u, 0x4440u + (i & 3));
        if (YCBCR && NCH >= 3) {
          const int Y = ch[0], cb = 2 * ch[1] - 255, cr = 2 * ch[NCH >= 3 ? 2 : 0] - 255;
          const int G = Y - ((cb + cr + 2) >> 2);
          ch[0] = clamp255(G + cr);
          ch[1] = clamp255(G);
          ch[NCH >= 3 ? 2 : 0] = clamp255(G + cb);
        }
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
          const int k = i * NCH + c;
          ow[k >> 2] |= (uint32_t)ch[c] << (8 * (k & 3));
        }
      }
      uint8_t *p = img + ((size_t)(8 * v + y) * g.w + (size_t)u * 8) * ctotal + cbase;
      if (aligned) {
        uint2 *q = reinterpret_cast<uint2 *>(p);
#pragma unroll
        for (int k = 0; k < NCH; ++k) q[k] = make_uint2(ow[2 * k], ow[2 * k + 1]);
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i)
          if (i < bw)
#pragma unroll
            for (int c = 0; c < NCH; ++c) {
              const int k = i * NCH + c;
              p[i * ctotal + c] = (uint8_t)(ow[k >> 2] >> (8 * (k & 3)));
            }
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// K-inv of a scaled decode (factor F = 2^lf, lf in 1..3): k_inverse's transform, then the final pixels of the thread's
// block (after the clamp and the inverse colour map) are box-averaged over the F x F windows that start at multiples
// of F -- each lies inside one block, so no thread needs another's pixels.  Windows on the right and bottom image
// edges are clipped: out = (S + n / 2) / n over the n pixels inside the image (1 <= n <= 64).
// Image z's output is [ceil(h / F)][ceil(w / F)][ctotal] at pixels + z * its size, or, with MIXED, at
// pixels + px_off[z] with its own geometry.  Grid, channel groups (cbase / ctotal) and MIXED as k_inverse.
// ---------------------------------------------------------------------------------------------
template <int NCH, bool MIXED = false>
__global__ void __launch_bounds__(kTile)
    k_inverse_scaled(const uint8_t *__restrict__ planes, const uint8_t *__restrict__ R, Geom g,
                     const DecTables *__restrict__ tabs, unsigned long long tab_stride, uint8_t *__restrict__ pixels,
                     int cbase, int ctotal, int lf, MixedDims md = {}, const unsigned long long *__restrict__ px_off = nullptr) {
  __shared__ int16_t sUn[256];
  __shared__ uint8_t sShift[2][64];
  __shared__ uint32_t sOut[NCH][kTile][17];  // per channel: the 64 pixel bytes of each thread's block (+1 pad)
  const Geom gb = g;  // bounding geometry (slot strides)
  if (MIXED && (!image_geom(md, blockIdx.z, g) || (int)blockIdx.y >= g.rows || (int)blockIdx.x * kTile >= g.cols)) return;
  const DecTables *T = reinterpret_cast<const DecTables *>(reinterpret_cast<const char *>(tabs) + (size_t)blockIdx.z * tab_stride);
  for (int i = threadIdx.x; i < 256; i += blockDim.x) sUn[i] = T->full_unmap[i];
  for (int i = threadIdx.x; i < 128; i += blockDim.x) sShift[i >> 6][i & 63] = T->shift[i >> 6][i & 63];
  const bool YCBCR = T->ycbcr != 0 && cbase == 0;  // (only the first three channels of an image are colour mapped)
  __syncthreads();
  const int v = blockIdx.y, u = blockIdx.x * kTile + threadIdx.x;
  if (u >= g.cols) return;
  const int bh = min(8, g.h - 8 * v), bw = min(8, g.w - 8 * u);
  const uint8_t *seg = planes + (size_t)blockIdx.z * gb.planes_bytes + (size_t)v * g.seg;

  // ---- the transform of k_inverse, clamped samples to sOut
#pragma unroll 1
  for (int c = 0; c < NCH; ++c) {
    int x[64];
    const uint8_t *src = seg + (size_t)(cbase + c) * g.cols * 64 + u;
    const uint8_t *sh = sShift[(YCBCR && NCH >= 3 && (c == 1 || c == 2)) ? 1 : 0];
#pragma unroll
    for (int j = 0; j < 64; ++j) {
      const int code = __ldg(src + (size_t)scan_pos(j) * g.cols);
      x[j] = (int)(short)(sUn[code] * (1 << sh[j]));
    }
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      wht8(x[r * 8 + 0], x[r * 8 + 1], x[r * 8 + 2], x[r * 8 + 3], x[r * 8 + 4], x[r * 8 + 5], x[r * 8 + 6], x[r * 8 + 7]);
#pragma unroll
      for (int i = 0; i < 8; ++i) x[r * 8 + i] >>= 3;
    }
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      wht8(x[q], x[8 + q], x[16 + q], x[24 + q], x[32 + q], x[40 + q], x[48 + q], x[56 + q]);
#pragma unroll
      for (int i = 0; i < 8; ++i) x[i * 8 + q] >>= 3;
    }
    {
      const uint8_t *Rp = MIXED ? R + (size_t)blockIdx.z * ctotal * gb.rows * gb.cols + (size_t)(cbase + c) * g.rows * g.cols
                                : R + ((size_t)blockIdx.z * ctotal + cbase + c) * g.rows * g.cols;
      const LowCorners k = load_corners(Rp, g, u, v);
      int lf9[9], rt9[9];
      nine(k.x11, k.x21, lf9);
      nine(k.x12, k.x22, rt9);
#pragma unroll
      for (int y = 0; y < 8; ++y) {
        int t[9];
        nine(lf9[y], rt9[y], t);
#pragma unroll
        for (int i = 0; i < 8; ++i) x[y * 8 + i] = clamp255((int)(short)(x[y * 8 + i] + t[i]));
      }
    }
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      const uint32_t lo = __byte_perm((uint32_t)x[4 * k], (uint32_t)x[4 * k + 1], 0x0040);
      const uint32_t hi = __byte_perm((uint32_t)x[4 * k + 2], (uint32_t)x[4 * k + 3], 0x0040);
      sOut[c][threadIdx.x][k] = __byte_perm(lo, hi, 0x5410);
    }
  }

  // ---- inverse colour map in place (a thread only touches its own block's bytes)
  uint8_t *px[NCH];  // pixel p = 8 * row + column of channel c: px[c][p]
#pragma unroll
  for (int c = 0; c < NCH; ++c) px[c] = reinterpret_cast<uint8_t *>(&sOut[c][threadIdx.x][0]);
  if (NCH >= 3 && YCBCR) {
#pragma unroll 4
    for (int p = 0; p < 64; ++p) {
      const int Y = px[0][p], cb = 2 * px[1][p] - 255, cr = 2 * px[NCH >= 3 ? 2 : 0][p] - 255;
      const int G = Y - ((cb + cr + 2) >> 2);
      px[0][p] = (uint8_t)clamp255(G + cr);
      px[1][p] = (uint8_t)clamp255(G);
      px[NCH >= 3 ? 2 : 0][p] = (uint8_t)clamp255(G + cb);
    }
  }

  // ---- box averages of the windows inside the image
  const int f = 1 << lf;
  const size_t ow = (size_t)((g.w + f - 1) >> lf), oh = (size_t)((g.h + f - 1) >> lf);
  uint8_t *img = MIXED ? pixels + px_off[blockIdx.z] : pixels + (size_t)blockIdx.z * ow * oh * ctotal;
  const int nwy = (bh + f - 1) >> lf, nwx = (bw + f - 1) >> lf;
#pragma unroll 1
  for (int wy = 0; wy < nwy; ++wy) {
    const int ny = min(f, bh - wy * f);
    uint8_t *row = img + (((size_t)(8 * v >> lf) + wy) * ow + (size_t)(8 * u >> lf)) * ctotal + cbase;
#pragma unroll 1
    for (int wx = 0; wx < nwx; ++wx) {
      const int nx = min(f, bw - wx * f), n = nx * ny, p0 = wy * f * 8 + wx * f;
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        int S = 0;
        for (int yy = 0; yy < ny; ++yy)
          for (int xx = 0; xx < nx; ++xx) S += px[c][p0 + yy * 8 + xx];
        row[(size_t)wx * ctotal + c] = (uint8_t)((S + (n >> 1)) / n);
      }
    }
  }
}

}  // namespace himgcu

#endif  // HIMG_B200_XFORM_KERNELS_CUH_
