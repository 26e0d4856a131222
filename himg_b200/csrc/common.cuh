// Shared device helpers for the B200 HIMG kernels (sm_100a only).
#ifndef HIMG_B200_COMMON_CUH_
#define HIMG_B200_COMMON_CUH_

#include <cuda_runtime.h>
#include <stdint.h>

namespace himgcu {

constexpr int kSyms = 261;
constexpr int kMaxNodes = 2 * kSyms - 1;
constexpr int kMaxRun = 16662;
constexpr int kTreeBytesMax = 360;  // ((2 + 9) * 261 + 7) / 8 = 359, rounded up

// Geometry of one image shape; identical for every image of a batch.
struct Geom {
  int w, h, nch, pstride;  // pstride = bytes between pixels of the INPUT (>= nch)
  int rows, cols;          // 8x8 blocks
  int mrows, mcols;        // 16x16 macroblocks of the low-res image
  int seg;                 // FRES segment = one block row of all channels = cols*64*nch bytes (<= 2^26: shape_ok)
  int lres_ch;             // mrows*mcols + rows*cols
  int lres_size;           // lres_ch * nch
  unsigned long long img_bytes;     // w*h*pstride
  unsigned long long out_img_bytes; // w*h*nch
  unsigned long long lres_stride;   // lres_size rounded up to 64
  unsigned long long planes_bytes;  // rows*seg
};

// Quantiser parameters travel as a __grid_constant__ kernel argument so that, with fully
// unrolled coefficient loops, shift/round become constant-bank operands (no extra instruction).
struct QuantParams {
  int shift[2][64];  // [0] luma / alpha, [1] chroma
  int round[2][64];  // shift ? 1 << (shift-1) : 0
};

// Decoder-side tables of one image, recovered from its in-band LMAP / QCFG / FMAP chunks.
struct DecTables {
  int16_t low_unmap[256];   // code byte -> value (Mapper::UnmapFrom8Bit, mapper.h:33-35)
  int16_t full_unmap[256];
  uint8_t shift[2][64];     // [0] luma / alpha, [1] chroma
  int ycbcr;
  int pad;
};

__host__ __device__ constexpr int scan_pos(int j) {
  // Position of coefficient j (= 8*row + col) in the reference's L-shaped-shell scan
  // (common.cpp:13-22): shell k = max(row, col) starts at k*k; odd shells run down column k then
  // left along row k, even shells run right along row k then up column k.
  const int r = j >> 3, c = j & 7;
  const int k = r > c ? r : c;
  if (k & 1) return c == k ? k * k + r : k * k + k + (k - c);
  return r == k ? k * k + c : k * k + k + (k - r);
}

__host__ __device__ constexpr int scan_coef(int i) {
  // inverse of scan_pos: the coefficient (8*row + col) at scan position i
  for (int j = 0; j < 64; ++j)
    if (scan_pos(j) == i) return j;
  return 0;
}

__host__ __device__ inline Geom make_geom(int w, int h, int nch, int pstride) {
  Geom g;
  g.w = w;
  g.h = h;
  g.nch = nch;
  g.pstride = pstride;
  g.rows = (h + 7) >> 3;
  g.cols = (w + 7) >> 3;
  g.mrows = (g.rows + 15) / 16;
  g.mcols = (g.cols + 15) / 16;
  g.seg = g.cols * 64 * nch;
  g.lres_ch = g.mrows * g.mcols + g.rows * g.cols;
  g.lres_size = g.lres_ch * nch;
  g.img_bytes = (unsigned long long)w * h * pstride;
  g.out_img_bytes = (unsigned long long)w * h * nch;
  g.lres_stride = ((unsigned long long)g.lres_size + 63) & ~63ull;
  g.planes_bytes = (unsigned long long)g.rows * g.seg;
  return g;
}

// Mixed-geometry batch: image i is dims[2i] x dims[2i+1] (device memory), bounded by max_w x max_h.  Every
// per-image scratch buffer keeps the slot stride of the bounding geometry make_geom(max_w, max_h, nch); inside
// its slot an image is laid out with its own geometry.
struct MixedDims {
  const int32_t *dims;
  int max_w, max_h, nch;
};

// Geometry of image i of a mixed batch.  False when its dims are < 1 or exceed the bounds: the image is then
// HIMGCU_ERR_ARG and nothing of it is decoded or encoded (gi is a 1 x 1 placeholder).
__device__ __forceinline__ bool image_geom(const MixedDims &m, int i, Geom &gi) {
  const int w = m.dims[2 * i], h = m.dims[2 * i + 1];
  const bool ok = w >= 1 && h >= 1 && w <= m.max_w && h <= m.max_h;
  gi = make_geom(ok ? w : 1, ok ? h : 1, m.nch, m.nch);
  return ok;
}

__device__ __forceinline__ int clamp255(int x) { return min(max(x, 0), 255); }

// Region decode: origin (x, y) of image i's rw x rh rectangle (origins [n][2], device memory).  False when the
// rectangle does not lie inside the image (rw, rh >= 1 are checked on the host).
__device__ __forceinline__ bool region_origin(const int32_t *__restrict__ origins, int i, const Geom &g, int rw, int rh,
                                              int &x, int &y) {
  x = origins[2 * i];
  y = origins[2 * i + 1];
  return x >= 0 && y >= 0 && x <= g.w - rw && y <= g.h - rh;
}

// Scaled region decode (factor 2^lf): origin (x, y) of image i's rw x rh rectangle of the scaled image
// [ceil(h / 2^lf)][ceil(w / 2^lf)].  The rectangle reads the source pixels [x << lf, min((x + rw) << lf, w)) x
// [y << lf, min((y + rh) << lf, h)).  False when it does not lie inside the scaled image.
__device__ __forceinline__ bool region_origin_scaled(const int32_t *__restrict__ origins, int i, const Geom &g, int lf, int rw,
                                                     int rh, int &x, int &y) {
  x = origins[2 * i];
  y = origins[2 * i + 1];
  const int f = 1 << lf;
  return x >= 0 && y >= 0 && x <= ((g.w + f - 1) >> lf) - rw && y <= ((g.h + f - 1) >> lf) - rh;
}

// Sequency-ordered 8-point Walsh-Hadamard butterflies (hadamard.cpp:18-44), in place.
__device__ __forceinline__ void wht8(int &x0, int &x1, int &x2, int &x3, int &x4, int &x5, int &x6,
                                     int &x7) {
  const int a0 = x0 + x4, a1 = x1 + x5, a2 = x2 + x6, a3 = x3 + x7;
  const int a4 = x0 - x4, a5 = x1 - x5, a6 = x2 - x6, a7 = x3 - x7;
  const int b0 = a0 + a2, b1 = a1 + a3, b2 = a0 - a2, b3 = a1 - a3;
  const int b4 = a4 + a6, b5 = a5 + a7, b6 = a4 - a6, b7 = a5 - a7;
  x0 = b0 + b1;
  x1 = b4 + b5;
  x2 = b6 + b7;
  x3 = b2 + b3;
  x4 = b2 - b3;
  x5 = b6 - b7;
  x6 = b4 - b5;
  x7 = b0 - b1;
}

// Nine-tap recursive midpoint interpolation (downsampled.cpp:116-169): t0=a, t8=b.
__device__ __forceinline__ void nine(int a, int b, int (&t)[9]) {
  t[0] = a;
  t[8] = b;
  t[4] = (t[0] + t[8] + 1) >> 1;
  t[2] = (t[0] + t[4] + 1) >> 1;
  t[6] = (t[4] + t[8] + 1) >> 1;
  t[1] = (t[0] + t[2] + 1) >> 1;
  t[3] = (t[2] + t[4] + 1) >> 1;
  t[5] = (t[4] + t[6] + 1) >> 1;
  t[7] = (t[6] + t[8] + 1) >> 1;
}

// Block-wide exclusive prefix sum of one uint32 per thread.  `warp_sums` needs blockDim/32 + 1
// entries of shared memory.  Returns the exclusive prefix; *total receives the block total.
__device__ __forceinline__ uint32_t block_exscan_u32(uint32_t v, uint32_t *warp_sums, uint32_t *total) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  uint32_t inc = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t t = __shfl_up_sync(0xffffffffu, inc, d);
    if (lane >= d) inc += t;
  }
  __syncthreads();  // protect warp_sums from a previous use
  if (lane == 31) warp_sums[wid] = inc;
  __syncthreads();
  if (wid == 0) {
    uint32_t s = lane < nw ? warp_sums[lane] : 0u;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, s, d);
      if (lane >= d) s += t;
    }
    if (lane < nw) warp_sums[lane] = s;  // inclusive per warp
  }
  __syncthreads();
  const uint32_t base = wid ? warp_sums[wid - 1] : 0u;
  *total = warp_sums[nw - 1];
  return base + inc - v;
}

}  // namespace himgcu

#endif  // HIMG_B200_COMMON_CUH_
