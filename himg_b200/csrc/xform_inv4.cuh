// K-inv, fast path (v4): the roofline kernel of the decoder.
//
// Same arithmetic as k_inverse (xform_kernels.cuh): gather + dequantise + inverse WHT with a floor
// >>3 after each pass + low-res add + clamp + inverse colour map (decoder.cpp:366-423,
// quantize.cpp:153-165, hadamard.cpp:90-103, ycbcr.cpp:54-82).  The kernel is bound by the integer
// (ALU) pipe, which accepts one warp instruction every other cycle, so the work is steered to the
// FMA pipe (IMAD / IDP) wherever an instruction exists there:
//
//  * WARP TILES: a warp owns 32 consecutive block pairs of the image in row-major order (whatever the
//    image width: no idle lanes on 1080p / 4K), stages their codes into its own shared-memory tile of
//    [nch * 64 scan positions][32 pairs x 2 codes] with its own cp.async group, and never synchronises
//    with the other warps of the CTA: while one warp waits for its codes the others compute, and the
//    LSU-, FMA- and ALU-heavy phases of different warps overlap (see the kernel);
//  * a thread owns two horizontally adjacent blocks as biased 16-bit lane pairs (exact while every
//    dequantised coefficient lies in [-4096, 4095]; the warp votes and otherwise redoes the channel
//    in int32 -- bit-exact either way, see v3);
//  * dequantisation: the two codes of a lane pair arrive as ONE 16-bit load; each table address is
//    ONE dp4a (byte * 2 + table base of the coefficient's shift: byte extraction, scaling and the
//    add in a single FMA-pipe instruction); the table holds (int16)(unmap << s) + 4096;
//  * the low-res corners are loaded by the owning thread while the tile is in flight;
//  * low-res add + clamp is one DPX instruction per lane pair, so is every output of the inverse
//    colour map; finished samples overwrite the thread's own codes in the tile.
//
// k_inverse4<NCH, TP, LF> also decodes scaled by 2^LF (LF 1..3), averaging inside the output phase.
//
// Preconditions (host checked, else k_inverse2 / k_inverse): cols % 16 == 0, height % 8 == 0,
// 16-byte aligned planes / pixels (LF > 0: 16 >> LF bytes), 2-byte aligned low-res image, nch in {1, 3}.
#ifndef HIMG_B200_XFORM_INV4_CUH_
#define HIMG_B200_XFORM_INV4_CUH_

#include "common.cuh"
#include "xform_lane.cuh"  // mid2 / nine2 / ibfly / smem_u32 / cp_async16

namespace himgcu {

// Block pairs (= threads) per CTA.  Two CTAs of 256 threads per SM leave 128 registers per thread; the
// gray kernel (no colour stage) fits 85 and runs three CTAs (8192^2 gray: 58 -> 54 us).  (Nine
// warps of RGB would still fit the shared memory of an SM -- 110 592 bytes of codes + 4 608 of tables is
// exactly half of it -- but at the 96 registers that leaves the kernel measured 17 % slower.)
constexpr int kInv4ThreadsRgb = 256, kInv4ThreadsGray = 256;

// 8-point sequency-ordered WHT on lane pairs whose bias is B on entry, followed by a floor shift by
// SH (0: none).  The bias on exit is 8 * B >> SH; no lane may leave 16 bits before the shift.
template <uint32_t B, int SH>
__device__ __forceinline__ void iwht8q(uint32_t &x0, uint32_t &x1, uint32_t &x2, uint32_t &x3, uint32_t &x4, uint32_t &x5,
                                       uint32_t &x6, uint32_t &x7) {
  constexpr uint32_t K1 = 2 * B * 0x00010001u, K2 = 4 * B * 0x00010001u, K3 = 8 * B * 0x00010001u;
  constexpr uint32_t M = (0xffffu >> SH) * 0x00010001u;
  uint32_t a0, a1, a2, a3, a4, a5, a6, a7, b0, b1, b2, b3, b4, b5, b6, b7;
  ibfly<K1>(x0, x4, a0, a4);
  ibfly<K1>(x1, x5, a1, a5);
  ibfly<K1>(x2, x6, a2, a6);
  ibfly<K1>(x3, x7, a3, a7);
  ibfly<K2>(a0, a2, b0, b2);
  ibfly<K2>(a1, a3, b1, b3);
  ibfly<K2>(a4, a6, b4, b6);
  ibfly<K2>(a5, a7, b5, b7);
  ibfly<K3>(b0, b1, x0, x7);
  ibfly<K3>(b4, b5, x1, x6);
  ibfly<K3>(b6, b7, x2, x5);
  ibfly<K3>(b2, b3, x3, x4);
  if (SH) {
    x0 = (x0 >> SH) & M;
    x1 = (x1 >> SH) & M;
    x2 = (x2 >> SH) & M;
    x3 = (x3 >> SH) & M;
    x4 = (x4 >> SH) & M;
    x5 = (x5 >> SH) & M;
    x6 = (x6 >> SH) & M;
    x7 = (x7 >> SH) & M;
  }
}

// 8-point sequency-ordered WHT on lane pairs WITHOUT bias constants: a packed word is the 32-bit integer
// hi * 65536 + lo with SIGNED fields, sums and differences of such words are exact modulo 2^32 whatever
// the signs of the fields, and every butterfly is a plain two-input add or subtract that either the ALU
// or the FMA pipe (IMAD) can execute.  The fields only have to be non-negative where a word is taken
// apart again (floor shift, DPX clamp); the caller arranges that through the DC input (see the kernel).
__device__ __forceinline__ void iwht8u(uint32_t &x0, uint32_t &x1, uint32_t &x2, uint32_t &x3, uint32_t &x4, uint32_t &x5,
                                       uint32_t &x6, uint32_t &x7) {
  const uint32_t a0 = x0 + x4, a1 = x1 + x5, a2 = x2 + x6, a3 = x3 + x7;
  const uint32_t a4 = x0 - x4, a5 = x1 - x5, a6 = x2 - x6, a7 = x3 - x7;
  const uint32_t b0 = a0 + a2, b1 = a1 + a3, b2 = a0 - a2, b3 = a1 - a3;
  const uint32_t b4 = a4 + a6, b5 = a5 + a7, b6 = a4 - a6, b7 = a5 - a7;
  x0 = b0 + b1;
  x1 = b4 + b5;
  x2 = b6 + b7;
  x3 = b2 + b3;
  x4 = b2 - b3;
  x5 = b6 - b7;
  x6 = b4 - b5;
  x7 = b0 - b1;
}

__device__ __forceinline__ uint32_t lds_u16(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}

// Dequantisation tables of one image, built once per image by k_inv_tables and copied into shared
// memory by every CTA of K-inv (the tables travel in-band, so they differ from image to image).
//   dq[slot(s)][code] = ((int16)(unmap[code] << s) >> pre) + bias       (quantize.cpp:153-165)
// One table per DISTINCT shift of the image, at most kInvSlots of them (a quality setting uses about five;
// the shared memory this saves against 16 tables is what lets a CTA of K-inv carry a ninth warp).  An
// image with more distinct shifts is decoded in OVERFLOW mode: slot 0 holds the plain unmap table, toff
// holds twice the shifts, and every warp takes the int32 path.
// When every shift of the image is >= 3 (any quality up to ~60) all coefficients are multiples of 8 and
// the row pass needs no floor at all: pre = 3, the tables hold value / 8 with a bias of 512 and the row
// pass skips its shift + mask.  Otherwise pre = 0 and the bias is 4096.
constexpr int kInvSlots = 8;
struct alignas(16) InvTables {
  uint16_t dq[kInvSlots][256];
  uint32_t toff[2][64];  // byte offset of the table of coefficient j (class luma / chroma) inside dq
  int pre, bias, ycbcr, overflow;
};
constexpr int kInvTableBytes = kInvSlots * 256 * 2 + 2 * 64 * 4;  // what a CTA copies (dq + toff)

// grid n, block 256.  (Shift bytes are masked: a rejected stream leaves its DecTables unspecified.)
__global__ void k_inv_tables(const DecTables *__restrict__ tabs, unsigned long long tab_stride, InvTables *__restrict__ out) {
  __shared__ int s_slot[16], s_nslots;
  const DecTables *T = reinterpret_cast<const DecTables *>(reinterpret_cast<const char *>(tabs) + (size_t)blockIdx.x * tab_stride);
  InvTables *O = out + blockIdx.x;
  const int t = threadIdx.x;
  const int mine = t < 128 ? (T->shift[t >> 6][t & 63] & 15) : 15;
  const bool pre3 = __syncthreads_and(mine >= 3) != 0;
  // slots of the shifts in use, in increasing order of the shift
  unsigned used = t < 128 ? 1u << mine : 0u;
#pragma unroll
  for (int d = 16; d >= 1; d >>= 1) used |= __shfl_xor_sync(0xffffffffu, used, d);
  if (t < 16) s_slot[t] = 0;
  if (t == 0) s_nslots = 0;
  __syncthreads();
  if ((t & 31) == 0 && t < 128) atomicOr(&s_slot[0], (int)used);  // (s_slot[0] doubles as the mask accumulator)
  __syncthreads();
  const unsigned mask = (unsigned)s_slot[0];
  __syncthreads();
  if (t < 16) s_slot[t] = __popc(mask & ((1u << t) - 1u));
  if (t == 0) s_nslots = __popc(mask);
  __syncthreads();
  const bool overflow = s_nslots > kInvSlots;
  const int pre = pre3 ? 3 : 0, bias = pre3 ? 512 : 4096;
  const int un = T->full_unmap[t];
  if (overflow) {
    O->dq[0][t] = (uint16_t)un;
  } else {
    for (int s = 0; s < 16; ++s)
      if (mask >> s & 1u) O->dq[s_slot[s]][t] = (uint16_t)(((int)(short)(un << s) >> pre) + bias);
  }
  // (overflow: twice the shift -- the table gather of the lane-pair path still runs and needs even, in-range offsets)
  if (t < 128) O->toff[t >> 6][t & 63] = overflow ? (uint32_t)mine * 2u : (uint32_t)s_slot[mine] * 512u;
  if (t == 0) {
    O->pre = pre;
    O->bias = bias;
    O->ycbcr = T->ycbcr != 0 ? 1 : 0;
    O->overflow = overflow ? 1 : 0;
  }
}

// Nine-tap midpoint interpolation on lane pairs that CARRY the addend of the fused add + clamp: every
// input and output lane is low-res | 0xf000 (= low-res - 4096 as int16).  The two 0xf000 of a sum always
// carry out of the low lane, so the rounding constant of the high lane is that carry (C = 1, not
// 0x00010001); the mask of the shifted sum takes its 0xf000 back in the same three-input logic operation.
// M = 0xf000f000 in a REGISTER the compiler cannot fold (a logic instruction takes one immediate only:
// with two immediates the mask and the OR are two instructions).
__device__ __forceinline__ uint32_t mid2m(uint32_t a, uint32_t b, uint32_t M) {
  return (((a + b + 1u) >> 1) & 0x00ff00ffu) | M;
}
__device__ __forceinline__ void nine2m(uint32_t a, uint32_t b, uint32_t M, uint32_t (&t)[9]) {
  t[0] = a;
  t[8] = b;
  t[4] = mid2m(a, b, M);
  t[2] = mid2m(a, t[4], M);
  t[6] = mid2m(t[4], b, M);
  t[1] = mid2m(a, t[2], M);
  t[3] = mid2m(t[2], t[4], M);
  t[5] = mid2m(t[4], t[6], M);
  t[7] = mid2m(t[6], b, M);
}

// int32 redo of one channel of a thread's two blocks (some lane of the warp left [-4096, 4095]).
// Reads the codes again; writes the clamped samples over them.
__device__ __noinline__ void inv4_wide(uint8_t *cc, int pitch, const uint32_t *tab, uint32_t dq_base, uint32_t top, uint32_t bot,
                                        int tab_bias, int pre, bool overflow) {
#pragma unroll 1
  for (int blk = 0; blk < 2; ++blk) {
    int y32[64];
#pragma unroll
    for (int j = 0; j < 64; ++j) {
      const uint32_t code = cc[scan_pos(j) * pitch + blk];
      if (overflow) y32[j] = (int)(short)((int)(short)lds_u16(dq_base + 2 * code) << (tab[j] >> 1));  // plain unmap table, tab = 2 * shift
      else y32[j] = (int)(short)(lds_u16(dq_base + tab[j] + 2 * code) - tab_bias) << pre;  // exact: the low bits were zeros
    }
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      wht8(y32[r * 8 + 0], y32[r * 8 + 1], y32[r * 8 + 2], y32[r * 8 + 3], y32[r * 8 + 4], y32[r * 8 + 5], y32[r * 8 + 6],
           y32[r * 8 + 7]);
#pragma unroll
      for (int i = 0; i < 8; ++i) y32[r * 8 + i] >>= 3;
    }
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      wht8(y32[q], y32[8 + q], y32[16 + q], y32[24 + q], y32[32 + q], y32[40 + q], y32[48 + q], y32[56 + q]);
#pragma unroll
      for (int i = 0; i < 8; ++i) y32[i * 8 + q] >>= 3;
    }
    int lf[9], rt[9];
    nine((int)((top >> (8 * blk)) & 0xffu), (int)((bot >> (8 * blk)) & 0xffu), lf);
    nine((int)((top >> (8 * blk + 8)) & 0xffu), (int)((bot >> (8 * blk + 8)) & 0xffu), rt);
#pragma unroll
    for (int y = 0; y < 8; ++y) {
      int tl[9];
      nine(lf[y], rt[y], tl);
#pragma unroll
      for (int i = 0; i < 8; ++i)
        cc[(y * 8 + i) * pitch + blk] = (uint8_t)__vimin_s32_relu((int)(short)(y32[y * 8 + i] + tl[i]), 255);
    }
  }
}

// Low-res corners (u, u+1, u+2) x (v, v+1) of a thread's block pair, edge clamped; u and cols are even.
template <int NCH>
__device__ __forceinline__ void inv4_corners(const uint8_t *__restrict__ R, int item, const Geom &g, int v, int u,
                                             uint32_t (&top)[NCH], uint32_t (&bot)[NCH]) {
  const int v2 = min(v + 1, g.rows - 1), u2 = min(u + 2, g.cols - 1);
#pragma unroll
  for (int c = 0; c < NCH; ++c) {
    const uint8_t *Rc = R + ((size_t)item * NCH + c) * g.rows * g.cols;
    const uint8_t *r0 = Rc + (size_t)v * g.cols, *r1 = Rc + (size_t)v2 * g.cols;
    top[c] = (uint32_t)__ldg(reinterpret_cast<const uint16_t *>(r0 + u)) | ((uint32_t)__ldg(r0 + u2) << 16);
    bot[c] = (uint32_t)__ldg(reinterpret_cast<const uint16_t *>(r1 + u)) | ((uint32_t)__ldg(r1 + u2) << 16);
  }
}

// Pixel row y of a block pair (wa: the 8 * NCH bytes of block A, wb: those of block B) to dst0 + y * row_bytes
// as 16-byte stores: whole pairs of a whole image.
template <int NCH>
struct Inv4Store16 {
  uint8_t *dst0;
  size_t row_bytes;
  __device__ __forceinline__ void operator()(int y, const uint32_t (&wa)[2 * NCH], const uint32_t (&wb)[2 * NCH]) const {
    uint4 *dst = reinterpret_cast<uint4 *>(dst0 + (size_t)y * row_bytes);
    if (NCH == 1) {
      dst[0] = make_uint4(wa[0], wa[1], wb[0], wb[1]);
    } else {
      dst[0] = make_uint4(wa[0], wa[1], wa[2], wa[3]);
      dst[1] = make_uint4(wa[4], wa[5], wb[0], wb[1]);
      dst[2] = make_uint4(wb[2], wb[3], wb[4], wb[5]);
    }
  }
};

// Output row wy of a block pair's 1 / 2^LF scaled decode (p: the (8 >> LF) * NCH pooled lane pairs, pixel-major,
// channel-minor; low lanes block A, high lanes block B) to dst0 + wy * row_bytes: the K bytes of block A, then those of
// block B, as NCH stores of 16 >> LF bytes each (8, 4 or 2: the pair's output row starts at a multiple of that).
template <int NCH, int LF>
struct Inv4StorePooled {
  uint8_t *dst0;
  size_t row_bytes;
  __device__ __forceinline__ void operator()(int wy, const uint32_t (&p)[(8 >> LF) * NCH]) const {
    constexpr int K = (8 >> LF) * NCH, UB = 16 >> LF;  // bytes per block, bytes per store
    // byte b of the pair's output row (every lane holds a byte value)
    auto byte = [&](int b) -> uint32_t { return b < K ? (p[b] & 0xffu) : (p[b - K] >> 16); };
    uint8_t *dst = dst0 + (size_t)wy * row_bytes;
    uint32_t wd[(2 * K + 3) / 4];
#pragma unroll
    for (int k = 0; k < (2 * K + 3) / 4; ++k) {
      wd[k] = 0u;
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (4 * k + j < 2 * K) wd[k] |= byte(4 * k + j) << (8 * j);
    }
#pragma unroll
    for (int q = 0; q < NCH; ++q) {
      if (UB == 8) reinterpret_cast<uint2 *>(dst)[q] = make_uint2(wd[2 * q], wd[2 * q + 1]);
      else if (UB == 4) reinterpret_cast<uint32_t *>(dst)[q] = wd[q];
      else reinterpret_cast<uint16_t *>(dst)[q] = (uint16_t)(wd[q >> 1] >> (16 * (q & 1)));
    }
  }
};

// The inverse proper for ONE thread = one block pair: codes in the thread's two byte columns `col` of a
// shared-memory tile whose rows
// (scan positions, channel-major) are PITCH bytes apart; the image's tables in sDq / sTab; pixel row y of
// the pair goes out through store(y, ...) (active threads only).  No barrier inside.
template <int NCH, int PITCH, class STORE, int LF>
__device__ __forceinline__ void inv4_compute(uint8_t *col, const uint8_t *sDq, const uint32_t *sTab, int pre, int tab_bias,
                                             bool overflow, bool ycbcr, bool active, const uint32_t (&top)[NCH],
                                             const uint32_t (&bot)[NCH], const STORE &store, uint32_t one) {
#ifdef HIMG_FORCE_PRE3  // (instruction counting only)
  const bool pre3 = true;
#else
  const bool pre3 = pre == 3;
#endif
  const uint32_t wide_mask = pre3 ? 0xfc00fc00u : 0xe000e000u;  // a lane outside the table's narrow range
  const uint32_t dq_base = smem_u32(sDq);  // (table offsets -> shared-memory addresses: added at the lookups' base)
#pragma unroll 1
  for (int c = 0; c < NCH; ++c) {
    uint8_t *cc = col + c * 64 * PITCH;
    const uint32_t *tab = sTab + ((ycbcr && NCH >= 3 && (c == 1 || c == 2)) ? 64 : 0);
    uint32_t tp = top[0], bt = bot[0];
#pragma unroll
    for (int k = 1; k < NCH; ++k) {
      tp = c == k ? top[k] : tp;
      bt = c == k ? bot[k] : bt;
    }
    // ---- gather + dequantise both blocks (biased lanes), remember every bit that was ever set
    uint32_t x[64], seen = 0;
#pragma unroll
    for (int j4 = 0; j4 < 64; j4 += 4) {
      const uint4 tb = *reinterpret_cast<const uint4 *>(tab + j4);
      const uint32_t tbj[4] = {tb.x, tb.y, tb.z, tb.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int j = j4 + k;
        const uint32_t w = *reinterpret_cast<const uint16_t *>(cc + scan_pos(j) * PITCH);
        // (the table base is the uniform part of the load's address: no add per coefficient)
        const uint32_t a = *reinterpret_cast<const uint16_t *>(sDq + __dp4a(w, 0x00000002u, tbj[k]));  // table + 2 * code of block A
        const uint32_t b = *reinterpret_cast<const uint16_t *>(sDq + __dp4a(w, 0x00000200u, tbj[k]));  // table + 2 * code of block B
        x[j] = a + (b << 16);
      }
      seen |= (x[j4] | x[j4 + 1]) | (x[j4 + 2] | x[j4 + 3]);  // (two three-input ORs)
    }
    const bool narrow = !overflow && __all_sync(0xffffffffu, !active || (seen & wide_mask) == 0);
    if (narrow) {
      // The table lanes carry a bias B (512 / 4096) and the butterflies add none, so after a pass only
      // the DC output of each transform is biased (by 8 B per pass).  One constant on the DC input gives
      // every output of the 2-D transform the same +32768 per lane; the outputs that were biased already
      // wrap around and take 0x7fff8000 (= 32768 per lane minus the carry of the wrap) afterwards.
      if (pre3) {
        x[0] += 0x80008000u;
#pragma unroll
        for (int r = 0; r < 8; ++r)
          iwht8u(x[r * 8 + 0], x[r * 8 + 1], x[r * 8 + 2], x[r * 8 + 3], x[r * 8 + 4], x[r * 8 + 5], x[r * 8 + 6], x[r * 8 + 7]);
      } else {
#pragma unroll
        for (int r = 0; r < 8; ++r)
          iwht8q<4096, 3>(x[r * 8 + 0], x[r * 8 + 1], x[r * 8 + 2], x[r * 8 + 3], x[r * 8 + 4], x[r * 8 + 5], x[r * 8 + 6], x[r * 8 + 7]);
#pragma unroll
        for (int q = 0; q < 8; ++q) x[q] += 0x80008000u;  // (every lane is floor(..) + 4096 here)
      }
#pragma unroll
      for (int q = 0; q < 8; ++q) iwht8u(x[q], x[8 + q], x[16 + q], x[24 + q], x[32 + q], x[40 + q], x[48 + q], x[56 + q]);
      x[0] += 0x7fff8000u;
      if (!pre3) {
#pragma unroll
        for (int q = 1; q < 8; ++q) x[q] += 0x7fff8000u;
      }
#pragma unroll
      for (int j = 0; j < 64; ++j) x[j] = (x[j] >> 3) & 0x1fff1fffu;
      const uint32_t M = one * 0xf000f000u;  // (opaque to the compiler: stays in a register)
      uint32_t lf[9], rt[9];
      // (the 0xf0 bytes make every lane low-res | 0xf000: see nine2m)
      nine2m(__byte_perm(tp, 0xf0u, 0x4140), __byte_perm(bt, 0xf0u, 0x4140), M, lf);  // left columns: corners u | u+1
      nine2m(__byte_perm(tp, 0xf0u, 0x4241), __byte_perm(bt, 0xf0u, 0x4241), M, rt);  // right columns: u+1 | u+2
#pragma unroll
      for (int y = 0; y < 8; ++y) {
        uint32_t tl[9];
        nine2m(lf[y], rt[y], M, tl);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          // lane + (low-res - 4096), min 255, max 0: two samples per instruction
          const uint32_t px = __viaddmin_s16x2_relu(x[y * 8 + i], tl[i], 0x00ff00ffu);
          // (inactive threads own their two columns of the tile too: no guard needed)
          *reinterpret_cast<uint16_t *>(cc + (y * 8 + i) * PITCH) = (uint16_t)__byte_perm(px, 0u, 0x4420);
        }
      }
    } else {
      inv4_wide(cc, PITCH, tab, dq_base, tp, bt, tab_bias, pre, overflow);
    }
  }

  // ---- inverse colour map + interleave + 16-byte stores (a thread reads back its own two columns)
  // `one` is the number 1 as a kernel argument: a multiplication by a value the compiler cannot see
  // stays an IMAD, i.e. it runs on the FMA pipe instead of the (fuller) ALU pipe.
  {
    const bool do_colour = ycbcr && NCH >= 3;
    const uint32_t two = one + one, k256 = one << 8, neg1 = 0u - one;
    // The unpacking byte-permute gives Y a bias of 512 and Cb one of 256 per lane for free (constant bytes).
    // With hb = (Cb + 256 + Cr) >> 1 = ((Cb + Cr) >> 1) + 128 and (Cb + Cr + 2) >> 1 = ((Cb + Cr) >> 1) + 1:
    //   Gp = Y + 512 - hb = G + 257  (positive lanes),  R = Gp + (2 Cr - 512),  B = Gp + (2 (Cb + 256) - 1024)
    // where 2 Cr - 512 is negative whatever Cr is, so the packed multiply-add never carries between lanes.
    uint32_t bias[NCH];
#pragma unroll
    for (int c = 0; c < NCH; ++c) bias[c] = !do_colour ? 0u : c == 0 ? 0x02u : c == 1 ? 0x01u : 0u;
    uint32_t pool[LF ? (8 >> LF) * NCH : 1];  // (LF > 0) window sums of the output row in progress, per channel
#pragma unroll
    for (int y = 0; y < 8; ++y) {
      uint32_t s[8 * NCH];  // lane pairs in memory order: pixel-major, channel-minor
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int c = 0; c < NCH; ++c)
          s[i * NCH + c] = __byte_perm((uint32_t) * reinterpret_cast<const uint16_t *>(col + (c * 64 + y * 8 + i) * PITCH), bias[c], 0x4140);
      if (NCH >= 3 && do_colour) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          uint32_t *ch = s + i * NCH;
          const uint32_t hb = ((ch[1] + ch[NCH >= 3 ? 2 : 0]) >> 1) & 0x01ff01ffu;
          const uint32_t Gp = hb * neg1 + ch[0];
          const uint32_t cr = ch[NCH >= 3 ? 2 : 0] * two + 0xfe00fe00u;
          const uint32_t cb = ch[1] * two + 0xfc00fc00u;
          ch[0] = __viaddmin_s16x2_relu(Gp, cr, 0x00ff00ffu);
          ch[1] = __viaddmin_s16x2_relu(Gp, 0xfefffeffu, 0x00ff00ffu);
          ch[NCH >= 3 ? 2 : 0] = __viaddmin_s16x2_relu(Gp, cb, 0x00ff00ffu);
        }
      }
      if constexpr (LF == 0) {
        // words of block A and of block B: four consecutive lane pairs -> one word each (every lane is a
        // byte value, so s1 * 256 + s0 = A0 | A1 << 8 | B0 << 16 | B1 << 24)
        uint32_t wa[2 * NCH], wb[2 * NCH];
#pragma unroll
        for (int m = 0; m < 2 * NCH; ++m) {
          const uint32_t pq = s[4 * m + 1] * k256 + s[4 * m], q = s[4 * m + 3] * k256 + s[4 * m + 2];
          wa[m] = __byte_perm(pq, q, 0x5410);
          wb[m] = __byte_perm(pq, q, 0x7632);
        }
        if (active) store(y, wa, wb);
      } else {
        // scaled decode: box sums of the F x F windows on the lanes (at most 64 * 255 = 16320 per lane), then
        // (S + F * F / 2) >> 2 LF per lane; output row y >> LF goes out after the window's last pixel row
        constexpr int F = 1 << LF, OW = 8 >> LF;
        if ((y & (F - 1)) == 0) {
#pragma unroll
          for (int m = 0; m < OW * NCH; ++m) pool[m] = 0u;
        }
#pragma unroll
        for (int wx = 0; wx < OW; ++wx)
#pragma unroll
          for (int i = 0; i < F; ++i)
#pragma unroll
            for (int c = 0; c < NCH; ++c) pool[wx * NCH + c] += s[(wx * F + i) * NCH + c];
        if ((y & (F - 1)) == F - 1) {
#pragma unroll
          for (int m = 0; m < OW * NCH; ++m) pool[m] = ((pool[m] + (F * F / 2) * 0x00010001u) >> (2 * LF)) & 0x00ff00ffu;
          if (active) store(y >> LF, pool);
        }
      }
    }
  }
}

// grid (ceil(rows * cols / 2 / TP), 1, n), block TP: one tile of TP consecutive block pairs per CTA.
// dynamic smem: tile [NCH * 64][2 * TP] | dq tables [8][256] u16 | table offsets [2][64] u32
//
// The codes of the tile and the image's tables arrive by cp.async (the threads of a tile row copy 2 * TP
// contiguous bytes), the CTA meets at one barrier, then the warps run the three channels and the
// output phase WITHOUT further barriers: a thread only ever touches its own two byte columns of the tile,
// and the phases of the inverse load different pipes (LSU in the gather, FMA in the butterflies, ALU in
// the clamps), so warps that drift apart fill each other's gaps.
// (Measured and dropped: several tiles per CTA with the next tile prefetched into L2 or copied early from
// inside the output phase, and tiles owned by single warps -- all slower than fresh CTAs whose start-up
// overlaps the other resident CTA.)
//
// LF > 0 (1..3): the decode scaled by F = 2^LF, through the pooled output phase of inv4_compute.  Image z's output is
// [h >> LF][w >> LF][NCH] at pixels + z * its size (every window is whole on these shapes), each pixel the rounded box
// average of its F x F window; the stores are 16 >> LF bytes wide.
template <int NCH, int TP, int LF>
__global__ void __launch_bounds__(TP, NCH == 1 ? 3 : 2)
    k_inverse4(const uint8_t *__restrict__ planes, const uint8_t *__restrict__ R, Geom g,
               const InvTables *__restrict__ tabs, unsigned long long tab_stride, uint8_t *__restrict__ pixels, uint32_t one) {
  extern __shared__ __align__(128) uint8_t sPl[];
  constexpr int PITCH = 2 * TP, CPR = TP / 8;  // bytes per tile row, 16-byte chunks per tile row
  static_assert(TP % 32 == 0 && TP == 8 * CPR, "a CTA is 8 groups of one thread per chunk of a tile row");
  uint8_t *sDq = sPl + NCH * 64 * PITCH;
  uint32_t *sTab = reinterpret_cast<uint32_t *>(sDq + kInvSlots * 256 * 2);

  const int t = threadIdx.x;
  const int PR = g.cols >> 1, total = g.rows * PR;
  const int f0 = blockIdx.x * TP;
  const int nact = min(TP, total - f0);
  const uint8_t *ipl = planes + (size_t)blockIdx.z * g.planes_bytes;
  uint8_t *img = pixels + (size_t)blockIdx.z * (LF ? (size_t)(g.w >> LF) * (size_t)(g.h >> LF) * NCH : g.out_img_bytes);
  const InvTables *T = reinterpret_cast<const InvTables *>(reinterpret_cast<const char *>(tabs) + (size_t)blockIdx.z * tab_stride);
  // block row / first pair of the tile's first element: one division per CTA, everything else by
  // carrying (a tile spans few block rows unless the image is very narrow)
  // (a true division: a 32-bit reciprocal of PR is not exact for every tile start of every accepted shape)
  const int v0 = (int)((uint32_t)f0 / (uint32_t)PR), p0 = f0 - v0 * PR;
  auto locate = [&](int k, int &v, int &p) {  // element f0 + k of the image -> block row, pair in the row
    if (PR >= 32) {
      v = v0;
      p = p0 + k;
      while (p >= PR) {
        p -= PR;
        ++v;
      }
    } else {
      v = (f0 + k) / PR;
      p = f0 + k - v * PR;
    }
  };
  {
    // the image's tables, then the tile: thread -> 16-byte chunk t % CPR (8 pairs of ONE block row:
    // cols % 16 == 0) of the tile rows t / CPR + 8 i; the threads of a row copy 2 * TP contiguous bytes
    const uint4 *tsrc = reinterpret_cast<const uint4 *>(T);
    for (int i = t; i < kInvTableBytes / 16; i += TP) cp_async16(sDq + 16 * i, tsrc + i);
    const int cq = t % CPR, r0 = t / CPR;
    if (8 * cq < nact) {
      int vl, pl;
      locate(8 * cq, vl, pl);
      const uint8_t *src = ipl + (size_t)vl * g.seg + 2 * pl + (size_t)r0 * g.cols;
      uint8_t *dst = sPl + r0 * PITCH + cq * 16;
      const size_t rstep = (size_t)8 * g.cols;
#pragma unroll 8
      for (int i = 0; i < NCH * 8; ++i) {
        cp_async16(dst + i * 8 * PITCH, src);
        src += rstep;
      }
    }
  }
  const int pre = T->pre, tab_bias = T->bias;
  const bool overflow = T->overflow != 0;
  const bool ycbcr = T->ycbcr != 0;
  const bool active = t < nact;
  int v, p;
  locate(active ? t : 0, v, p);
  const int u = 2 * p;
  uint32_t top[NCH], bot[NCH];
  inv4_corners<NCH>(R, blockIdx.z, g, v, u, top, bot);
  cp_async_wait_all();
  __syncthreads();  // the only barrier: from here on a thread touches its own two byte columns only
  using Store = std::conditional_t<LF == 0, Inv4Store16<NCH>, Inv4StorePooled<NCH, LF>>;
  constexpr int OB = 8 >> LF;  // output pixels of a block per row
  const size_t ow = (size_t)(g.w >> LF);
  inv4_compute<NCH, PITCH, Store, LF>(sPl + 2 * t, sDq, sTab, pre, tab_bias, overflow, ycbcr, active, top, bot,
                                      Store{img + ((size_t)(OB * v) * ow + (size_t)u * OB) * NCH, ow * NCH}, one);
}

}  // namespace himgcu

#endif  // HIMG_B200_XFORM_INV4_CUH_
