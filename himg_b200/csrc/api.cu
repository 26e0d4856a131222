// C-ABI implementation (include/himg_cuda.h): context, device scratch, launch sequences.
// Product code: no CPU fallback; the test-only CPU restatement is never linked or called here.
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <type_traits>
#include <vector>

#include "../../include/himg_cuda.h"
#include "huff_dec_kernels.cuh"
#include "huff_enc_kernels.cuh"
#include "tables.h"
#include "xform_fwd3.cuh"
#include "xform_inv2.cuh"
#include "xform_avg2.cuh"
#include "xform_inv4.cuh"
#include "xform_kernels.cuh"
#include "xform_region.cuh"

using namespace himgcu;

namespace {

// dst may be page-locked host memory (unified addressing): the stores are visible to the host once an
// event recorded after the kernel has completed.
__global__ void k_store_u32(uint32_t *__restrict__ dst, const uint32_t *__restrict__ src, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = src[i];
}

struct DevBuf {
  void *p = nullptr;
  size_t cap = 0;
};

struct ProfRec {
  const char *name;
  cudaEvent_t a, b;
};

}  // namespace

struct himgcu_ctx {
  int device = 0;
  cudaStream_t own_stream = nullptr;
  cudaStream_t stream = nullptr;
  cudaStream_t in_stream = nullptr, out_stream = nullptr;  // copy streams of the host-buffer batch calls
  cudaStream_t aux_stream = nullptr;                       // second branch of a single-image decode
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  // The host-buffer batch calls keep up to kMaxLanes sub-batches in flight.  Lane 0 is this context;
  // lanes 1.. are child contexts (own stream, own workspace) so that the latency-bound kernels of one
  // sub-batch (tree construction, the low-res chunk) overlap the wide kernels of its neighbours.
  static constexpr int kMaxLanes = 8;
  std::vector<himgcu_ctx *> lanes;
  int host_lanes = 3;
  cudaEvent_t ev_in[kMaxLanes] = {}, ev_cmp[kMaxLanes] = {}, ev_out[kMaxLanes] = {};
  std::string err;
  std::map<std::string, DevBuf> bufs;
  DevBuf full_lut;  // 7616-byte |x| -> code LUT, uploaded once
  DevBuf signed_lut;  // 32 KiB signed LUT (index m + 16384) for k_forward3
  void *pinned = nullptr;
  size_t pinned_cap = 0;
  void *stage[2] = {nullptr, nullptr};  // page-locked staging slots of the single-image host calls
  cudaEvent_t stage_ev[2] = {nullptr, nullptr};
  bool profile = false;
  std::vector<ProfRec> pending;
  std::vector<cudaEvent_t> event_pool;
  std::map<std::string, std::pair<double, int>> prof;
  std::vector<std::string> prof_names;
  uint64_t launches = 0;
  size_t max_workspace = (size_t)24 << 30;
  int item_lists = 1;  // hand the item lists of the histogram pass to the packer (option "item_lists")
  // framed chunks without parts, option "huff_warp_teams": 1 = k_huff_hist4 / k_huff_pack4 when the batch has a
  // wave of segments, 2 = whenever possible (tests), 0 = never (k_huff_hist2 / k_huff_pack3)
  int huff_warp_teams = 1;
  size_t host_sub_bytes = (size_t)192 << 20;  // staged bytes per sub-batch of the host-buffer calls (measured best: 128-192 MB)
  bool force_generic = false;  // tests: route everything through the generic kernels
  int xform_variant = 0;       // experiments: 0 = newest fast kernels, 1 = previous generation
  // small table uploads are cached by key so that steady-state calls issue no host sync
  std::string lowres_key, prefix_key;
};

namespace {

int fail(himgcu_ctx *c, int code, const char *fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (c) c->err = buf;
  return code;
}

#define CK(call)                                                                              \
  do {                                                                                        \
    cudaError_t e_ = (call);                                                                  \
    if (e_ != cudaSuccess)                                                                    \
      return fail(ctx, HIMGCU_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                  __FILE__, __LINE__);                                                        \
  } while (0)

int ensure(himgcu_ctx *ctx, const char *name, size_t bytes, void **out) {
  DevBuf &b = ctx->bufs[name];
  if (b.cap < bytes) {
    if (b.p) {
      CK(cudaStreamSynchronize(ctx->stream));
      CK(cudaFree(b.p));
      b.p = nullptr;
      b.cap = 0;
    }
    const size_t want = (bytes + 255) & ~(size_t)255;
    CK(cudaMalloc(&b.p, want));
    b.cap = want;
    ctx->lowres_key.clear();
    ctx->prefix_key.clear();
  }
  *out = b.p;
  return HIMGCU_OK;
}

#define ENSURE(name, bytes, ptr)                                             \
  do {                                                                       \
    void *p_ = nullptr;                                                      \
    int rc_ = ensure(ctx, name, (bytes), &p_);                               \
    if (rc_ != HIMGCU_OK) return rc_;                                        \
    ptr = reinterpret_cast<decltype(ptr)>(p_);                               \
  } while (0)

cudaEvent_t get_event(himgcu_ctx *ctx) {
  if (!ctx->event_pool.empty()) {
    cudaEvent_t e = ctx->event_pool.back();
    ctx->event_pool.pop_back();
    return e;
  }
  cudaEvent_t e;
  cudaEventCreate(&e);
  return e;
}

struct LaunchScope {
  himgcu_ctx *ctx;
  const char *name;
  cudaEvent_t a = nullptr, b = nullptr;
  LaunchScope(himgcu_ctx *c, const char *n) : ctx(c), name(n) {
    ++ctx->launches;
    if (ctx->profile) {
      a = get_event(ctx);
      b = get_event(ctx);
      cudaEventRecord(a, ctx->stream);
    }
  }
  ~LaunchScope() {
    if (ctx->profile) {
      cudaEventRecord(b, ctx->stream);
      ctx->pending.push_back({name, a, b});
    }
  }
};

#define LAUNCH(name, kernel, grid, block, smem, ...)                                         \
  do {                                                                                       \
    {                                                                                        \
      LaunchScope ls_(ctx, name);                                                            \
      kernel<<<grid, block, smem, ctx->stream>>>(__VA_ARGS__);                               \
    }                                                                                        \
    cudaError_t e_ = cudaGetLastError();                                                     \
    if (e_ != cudaSuccess)                                                                   \
      return fail(ctx, HIMGCU_ERR_CUDA, "launch %s failed: %s", name, cudaGetErrorString(e_)); \
  } while (0)

void resolve_profile(himgcu_ctx *ctx) {
  for (ProfRec &r : ctx->pending) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) {
      auto it = ctx->prof.find(r.name);
      if (it == ctx->prof.end()) {
        ctx->prof[r.name] = {ms, 1};
        ctx->prof_names.push_back(r.name);
      } else {
        it->second.first += ms;
        it->second.second += 1;
      }
    }
    ctx->event_pool.push_back(r.a);
    ctx->event_pool.push_back(r.b);
  }
  ctx->pending.clear();
}

// A block row (FRES segment) holds at most kMaxSegBytes = 2^26 bytes, i.e. 8 * ceil(w / 8) * nch <= 2^23.  A token
// covers at least one byte and takes at most a 32-bit code plus 14 extra bits, so a segment codes to fewer than
// 46 * 2^26 < 2^32 bits: the segment sizes and the 32-bit bit counts and positions of the entropy kernels cannot
// overflow, and Geom::seg fits an int.
constexpr long long kMaxSegBytes = 1ll << 26;

bool shape_ok(int w, int h, int nch) {
  if (w < 1 || h < 1 || nch < 1 || nch > 255) return false;  // (the container stores the channel count in one byte)
  // (64-bit rounding: w + 7 and h + 7 overflow an int near 2^31)
  const unsigned long long px = (unsigned long long)w * h * nch;
  const long long rows = ((long long)h + 7) >> 3, seg = (((long long)w + 7) >> 3) * 64 * nch;
  return px < (1ull << 31) && rows <= 65535 && seg <= kMaxSegBytes;
}

int upload_full_lut(himgcu_ctx *ctx) {
  if (ctx->full_lut.p) return HIMGCU_OK;
  CK(cudaMalloc(&ctx->full_lut.p, kFullMapLutSize));
  ctx->full_lut.cap = kFullMapLutSize;
  CK(cudaMemcpyAsync(ctx->full_lut.p, FullMapLut(), kFullMapLutSize, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return HIMGCU_OK;
}

int upload_signed_lut(himgcu_ctx *ctx) {
  if (ctx->signed_lut.p) return HIMGCU_OK;
  std::vector<uint8_t> lut(2 * kLutCenter + 64, 0);  // padded: the kernel copies whole 16-byte words
  const uint8_t *mag = FullMapLut();
  for (int v = 0; v < 2 * kLutCenter; ++v) {
    const int m = v - kLutCenter, a = m < 0 ? -m : m;
    const int code = mag[a < kFullMapLutSize ? a : kFullMapLutSize - 1];  // >= 7608 -> 127
    lut[v] = (uint8_t)(m >= 0 ? code : (256 - code) & 0xff);
  }
  CK(cudaMalloc(&ctx->signed_lut.p, lut.size()));
  ctx->signed_lut.cap = lut.size();
  CK(cudaMemcpyAsync(ctx->signed_lut.p, lut.data(), lut.size(), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return HIMGCU_OK;
}

// dp4a weights of channel c (see ColourW): coef[k] multiplies byte k of the pixel.
//   Y  = (r + 2g + b + 2) >> 2          = byte 1 of 64 * (r + 2g + b + 2)
//   Cb = (b - g + 256) >> 1              = byte 1 of 128 * (b + (255 - g) + 1)     (g complemented by XOR)
//   Cr = (r - g + 256) >> 1              = byte 1 of 128 * (r + (255 - g) + 1)
//   plain channel                        = byte 0 of 1 * value
void make_colour(int nch, bool ycbcr, ColourW *cw) {
  for (int c = 0; c < 4; ++c) {
    uint32_t coef[4] = {0, 0, 0, 0}, add = 0, sel = 0x7430;
    bool xg = false;
    if (ycbcr && nch >= 3 && c < 3) {
      sel = 0x7531;
      add = 128;
      if (c == 0) { coef[0] = 64; coef[1] = 128; coef[2] = 64; }
      if (c == 1) { coef[1] = 128; coef[2] = 128; xg = true; }
      if (c == 2) { coef[0] = 128; coef[1] = 128; xg = true; }
    } else {
      coef[c] = 1;
    }
    ColourW &w = cw[c];
    w.add = add;
    w.sel = sel;
    w.has_xm = xg ? 1 : 0;
    for (int k = 0; k < 3; ++k) {  // word k of a row: bytes 4k .. 4k+3, channel = byte index % nch
      uint32_t m = 0;
      for (int by = 0; by < 4; ++by)
        if (xg && (4 * k + by) % nch == 1) m |= 0xffu << (8 * by);
      w.xm[k] = m;
    }
    for (int sh = 0; sh < 4; ++sh) {
      uint32_t w0 = 0, w1 = 0;
      for (int k = 0; k < nch && k < 4; ++k) {
        const int pos = sh + k;
        if (pos < 4) w0 |= coef[k] << (8 * pos);
        else w1 |= coef[k] << (8 * (pos - 4));
      }
      w.w0[sh] = w0;
      w.w1[sh] = w1;
    }
  }
}

bool make_quant_recs(const EncodeTables &t, Fwd3Params *P) {
  // value range after the shift: |T| <= 16320, so |m| <= (16320 + round) >> shift
  int half = 1;
  for (int cls = 0; cls < 2; ++cls)
    for (int j = 0; j < 64; ++j) {
      const int s = cls ? t.shift_chroma[j] : t.shift_luma[j];
      if (s > 14) return false;
      half = std::max(half, ((16320 + (s ? 1 << (s - 1) : 0)) >> s) + 1);
    }
  half = std::min((half + 63) & ~63, kLutCenter - 64);
  P->lut_half = half;
  for (int cls = 0; cls < 2; ++cls)
    for (int i = 0; i < 64; ++i) {
      const int j = scan_coef(i);  // records are stored in scan order
      const int s = cls ? t.shift_chroma[j] : t.shift_luma[j];
      const uint32_t rep = 0x00010001u;
      QuantRec &r = P->rec[cls][i];
      r.c2 = (s ? (1u << (s - 1)) - 1u : 0u) * rep;
      r.tmask = s ? rep : 0u;
      r.off = (uint32_t)(half - (16384 >> s));
      r.s16 = (uint32_t)s + 16u;
    }
  return true;
}

QuantParams make_quant(const EncodeTables &t) {
  QuantParams q;
  for (int j = 0; j < 64; ++j) {
    q.shift[0][j] = t.shift_luma[j];
    q.shift[1][j] = t.shift_chroma[j];
    q.round[0][j] = t.shift_luma[j] ? 1 << (t.shift_luma[j] - 1) : 0;
    q.round[1][j] = t.shift_chroma[j] ? 1 << (t.shift_chroma[j] - 1) : 0;
  }
  return q;
}

// ---- stage launchers (device pointers, asynchronous) -------------------------------------------
//
// The stage functions are instantiated for uniform batches (MIXED = false) and for batches of mixed geometry
// (MIXED = true, see MixedDims): g is then the bounding geometry, which sizes the scratch, `md` holds the images' own
// sizes, and image i's pixels start at d_pixels + px_off[i].  Uniform calls leave md and px_off at the kernels' own
// defaults.  A mixed batch always takes the generic kernels.

template <int N>
using Nch = std::integral_constant<int, N>;

// Calls launch(Nch<NCH>(), cbase, ctotal, ycbcr) for every channel group [cbase, cbase + NCH) of an nch-channel image:
// up to four channels are one group, more are the first three and then one group per further channel.  Only the group
// at channel 0 carries the colour map.
template <class F>
int for_channel_groups(int nch, bool ycbcr, F &&launch) {
  switch (nch) {
    case 1: return launch(Nch<1>(), 0, 1, false);
    case 2: return launch(Nch<2>(), 0, 2, false);
    case 3: return launch(Nch<3>(), 0, 3, ycbcr);
    case 4: return launch(Nch<4>(), 0, 4, ycbcr);
    default: break;
  }
  int rc = launch(Nch<3>(), 0, nch, ycbcr);
  for (int c = 3; c < nch && !rc; ++c) rc = launch(Nch<1>(), c, nch, false);
  return rc;
}

template <int NCH>
int launch_avg2(himgcu_ctx *ctx, const uint8_t *d_pixels, int n, const Geom &g, bool ycbcr, uint8_t *d_avg) {
  Avg2Params P;
  make_colour(g.nch, ycbcr, P.cw);
  dim3 grid((g.cols / 2 + kAvg2Threads - 1) / kAvg2Threads, g.rows, n);
  LAUNCH("k_lowres_avg", (k_lowres_avg2<NCH>), grid, kAvg2Threads, 0, d_pixels, g, P, d_avg);
  return HIMGCU_OK;
}

template <bool MIXED = false>
int stage_lowres(himgcu_ctx *ctx, const uint8_t *d_pixels, int n, const Geom &g, bool ycbcr, uint8_t *d_L,
                 const MixedDims &md = {}, const unsigned long long *px_off = nullptr) {
  uint8_t *d_avg;
  const size_t nlow = (size_t)n * g.nch * g.rows * g.cols;
  ENSURE("avg", nlow, d_avg);
  int rc;
  // lane-pair fast path: whole 16-pixel block pairs, tightly packed pixels, 16-byte aligned rows
  const bool fast = !MIXED && !ctx->force_generic && !(ctx->xform_variant & 1) && g.pstride == g.nch && (g.w % 16) == 0 &&
                    (reinterpret_cast<uintptr_t>(d_pixels) & 15) == 0 && (g.img_bytes & 15) == 0 &&
                    (reinterpret_cast<uintptr_t>(d_avg) & 1) == 0 && (g.nch == 1 || g.nch == 3 || g.nch == 4);
  if (fast) {
    switch (g.nch) {
      case 1: rc = launch_avg2<1>(ctx, d_pixels, n, g, false, d_avg); break;
      case 3: rc = launch_avg2<3>(ctx, d_pixels, n, g, ycbcr, d_avg); break;
      default: rc = launch_avg2<4>(ctx, d_pixels, n, g, ycbcr, d_avg); break;
    }
  } else {
    // cbase / ctotal: the channel group [cbase, cbase + NCH) of an image with ctotal channels (see k_lowres_avg)
    rc = for_channel_groups(g.nch, ycbcr, [&](auto nc, int cbase, int ctotal, bool yc) -> int {
      constexpr int NCH = decltype(nc)::value;
      const dim3 grid((g.cols + kTile - 1) / kTile, g.rows, n);
      if (yc)
        LAUNCH("k_lowres_avg", (k_lowres_avg<NCH, true, MIXED>), grid, kTile, 0, d_pixels + cbase, g, d_avg, cbase, ctotal, md,
               px_off);
      else
        LAUNCH("k_lowres_avg", (k_lowres_avg<NCH, false, MIXED>), grid, kTile, 0, d_pixels + cbase, g, d_avg, cbase, ctotal, md,
               px_off);
      return HIMGCU_OK;
    });
  }
  if (rc) return rc;
  const int threads = std::min(256, (g.cols + 31) & ~31);
  const dim3 grid((unsigned)(n * g.nch), (g.rows + kCompRows - 1) / kCompRows);
  LAUNCH("k_lowres_comp", k_lowres_comp<MIXED>, grid, threads, 0, d_avg, n * g.nch, g.rows, g.cols, d_L, md);
  return HIMGCU_OK;
}

int upload_lowres_tables(himgcu_ctx *ctx, const EncodeTables *enc, const int16_t *unmap, LowResTables **d_out) {
  LowResTables h;
  memset(&h, 0, sizeof(h));
  if (enc) {
    memcpy(h.map_lut, enc->low_map_lut, 256);
    for (int c = 0; c < 128; ++c) h.unmap[c] = (int16_t)enc->low_table[c];
    for (int k = 1; k <= 127; ++k) h.unmap[256 - k] = (int16_t)(-(int16_t)enc->low_table[k]);
    h.unmap[128] = h.unmap[129];
  } else {
    memcpy(h.unmap, unmap, sizeof(h.unmap));
  }
  LowResTables *d;
  ENSURE("lowres_tables", sizeof(LowResTables), d);
  const std::string key = enc ? "q" + std::to_string(enc->quality) : std::string();
  if (key.empty() || ctx->lowres_key != key) {
    CK(cudaMemcpyAsync(d, &h, sizeof(h), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));  // `h` lives on this stack frame
    ctx->lowres_key = key;
  }
  *d_out = d;
  return HIMGCU_OK;
}

template <bool MIXED = false>
int stage_lres_encode(himgcu_ctx *ctx, const uint8_t *d_L, int n, const Geom &g, const EncodeTables &t, uint8_t *d_lres,
                      const MixedDims &md = {}) {
  LowResTables *d_tabs;
  int rc = upload_lowres_tables(ctx, &t, nullptr, &d_tabs);
  if (rc) return rc;
  const long long nmb = (long long)n * g.nch * g.mrows * g.mcols;
  const unsigned blocks = (unsigned)((nmb + kLresWarps * 2 - 1) / (kLresWarps * 2));
  LAUNCH("k_lres_dpcm_enc", (k_lres_dpcm<true, MIXED>), blocks, kLresWarps * 32, 0, d_L, d_lres, (uint8_t *)nullptr, g, n,
         d_tabs->map_lut, d_tabs->unmap, (unsigned long long)0, md);
  return HIMGCU_OK;
}

template <int NCH, int COLS>
int launch_fwd3(himgcu_ctx *ctx, const uint8_t *d_pixels, const uint8_t *d_L, int n, const Geom &g, bool ycbcr,
                const Fwd3Params &P, uint8_t *d_planes) {
  const int total_pairs = g.rows * (g.cols / 2);
  const int tiles = (total_pairs + kFwd3Threads - 1) / kFwd3Threads;
  // consecutive tiles per CTA (the next tile loads under the tail of the current one): as many as
  // leave at least four waves of CTAs on the GPU, at most 8
  int tpc = (int)std::max<long long>(1, std::min<long long>(8, (long long)tiles * n / (148 * 2 * 4)));
  if (ctx->xform_variant & 4) tpc = 1;  // experiment
  dim3 grid((tiles + tpc - 1) / tpc, 1, n);
  const int smem = ((2 * P.lut_half + 1 + 127) & ~127) + kFwd3Threads * 8 * 16 * NCH;
  const uint8_t *lut = (const uint8_t *)ctx->signed_lut.p;
  if (NCH >= 3 && ycbcr) {
    constexpr bool Y = NCH >= 3;  // (no dead <1, true> instances)
    CK(cudaFuncSetAttribute((k_forward3<NCH, Y, COLS>), cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    LAUNCH("k_forward", (k_forward3<NCH, Y, COLS>), grid, kFwd3Threads, smem, d_pixels, d_L, g, P, lut, d_planes, tpc);
  } else {
    CK(cudaFuncSetAttribute((k_forward3<NCH, false, COLS>), cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    LAUNCH("k_forward", (k_forward3<NCH, false, COLS>), grid, kFwd3Threads, smem, d_pixels, d_L, g, P, lut, d_planes, tpc);
  }
  return HIMGCU_OK;
}

template <bool MIXED = false>
int stage_forward(himgcu_ctx *ctx, const uint8_t *d_pixels, const uint8_t *d_L, int n, const Geom &g,
                  const EncodeTables &t, uint8_t *d_planes, const MixedDims &md = {},
                  const unsigned long long *px_off = nullptr) {
  // fast path: whole 16-pixel-wide block pairs, tightly packed pixels, 16-byte aligned rows
  if (!MIXED && !ctx->force_generic && !(ctx->xform_variant & 1) && g.pstride == g.nch && (g.w % 16) == 0 && (g.h % 8) == 0 &&
      (reinterpret_cast<uintptr_t>(d_pixels) & 15) == 0 && (reinterpret_cast<uintptr_t>(d_L) & 1) == 0 &&
      (g.nch == 1 || g.nch == 3 || g.nch == 4)) {
    Fwd3Params P;
    if (make_quant_recs(t, &P)) {
      int rc = upload_signed_lut(ctx);
      if (rc) return rc;
      make_colour(g.nch, t.ycbcr, P.cw);
      // plane stride as an immediate for the common widths (1080p, 4K RGB; 8K gray)
      if (g.nch == 3 && g.cols == 240) return launch_fwd3<3, 240>(ctx, d_pixels, d_L, n, g, t.ycbcr, P, d_planes);
      if (g.nch == 3 && g.cols == 480) return launch_fwd3<3, 480>(ctx, d_pixels, d_L, n, g, t.ycbcr, P, d_planes);
      if (g.nch == 1 && g.cols == 1024) return launch_fwd3<1, 1024>(ctx, d_pixels, d_L, n, g, false, P, d_planes);
      switch (g.nch) {
        case 1: return launch_fwd3<1, 0>(ctx, d_pixels, d_L, n, g, false, P, d_planes);
        case 3: return launch_fwd3<3, 0>(ctx, d_pixels, d_L, n, g, t.ycbcr, P, d_planes);
        default: return launch_fwd3<4, 0>(ctx, d_pixels, d_L, n, g, t.ycbcr, P, d_planes);
      }
    }
  }
  int rc = upload_full_lut(ctx);
  if (rc) return rc;
  const QuantParams qp = make_quant(t);
  const uint8_t *lut = (const uint8_t *)ctx->full_lut.p;
  return for_channel_groups(g.nch, t.ycbcr, [&](auto nc, int cbase, int ctotal, bool yc) -> int {
    constexpr int NCH = decltype(nc)::value;
    const dim3 grid((g.cols + kTile - 1) / kTile, g.rows, n);
    if (yc)
      LAUNCH("k_forward", (k_forward<NCH, true, MIXED>), grid, kTile, 0, d_pixels + cbase, d_L, g, qp, lut, d_planes, cbase, ctotal,
             md, px_off);
    else
      LAUNCH("k_forward", (k_forward<NCH, false, MIXED>), grid, kTile, 0, d_pixels + cbase, d_L, g, qp, lut, d_planes, cbase,
             ctotal, md, px_off);
    return HIMGCU_OK;
  });
}

template <int NCH>
int launch_inv2(himgcu_ctx *ctx, const uint8_t *d_planes, const uint8_t *d_R, int n, const Geom &g,
                const DecTables *d_tabs, unsigned long long tab_stride, uint8_t *d_pixels) {
  // balanced column tiles of at most 256 blocks, multiples of 16 blocks
  const int nt = (g.cols + kInv2Pitch - 1) / kInv2Pitch;
  const int tile_cols = std::min(kInv2Pitch, (((g.cols + nt - 1) / nt) + 15) & ~15);
  dim3 grid((g.cols + tile_cols - 1) / tile_cols, g.rows, n);
  const int smem = NCH * 64 * kInv2Pitch + NCH * kInv2Threads * 17 * 4;
  CK(cudaFuncSetAttribute(k_inverse2<NCH>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  LAUNCH("k_inverse", (k_inverse2<NCH>), grid, kInv2Threads, smem, d_planes, d_R, g, d_tabs, tab_stride, tile_cols,
         d_pixels);
  return HIMGCU_OK;
}

// Dequantisation tables of the lane-pair kernels: one set per image of d_tabs (tab_stride apart), ntab of them.
int launch_inv_tables(himgcu_ctx *ctx, const DecTables *d_tabs, int ntab, unsigned long long tab_stride, InvTables **d_inv) {
  InvTables *d;
  ENSURE("inv_tables", (size_t)ntab * sizeof(InvTables), d);
  LAUNCH("k_inv_tables", k_inv_tables, ntab, 256, 0, d_tabs, tab_stride, d);
  *d_inv = d;
  return HIMGCU_OK;
}

// Lane-pair inverse: k_inverse4, or at LF > 0 k_inverse4_scaled (a decode scaled by 2^LF, same shapes and tiles).
template <int NCH, int LF>
int launch_inv4(himgcu_ctx *ctx, const uint8_t *d_planes, const uint8_t *d_R, int n, const Geom &g,
                const DecTables *d_tabs, unsigned long long tab_stride, uint8_t *d_pixels) {
  // per-image dequantisation tables first (the tables travel in-band); one set when the caller has one
  InvTables *d_inv;
  int rc = launch_inv_tables(ctx, d_tabs, tab_stride ? n : 1, tab_stride, &d_inv);
  if (rc) return rc;
  const unsigned long long inv_stride = tab_stride ? sizeof(InvTables) : 0;
  const int total_pairs = g.rows * (g.cols / 2);
  constexpr int TP = NCH == 1 ? kInv4ThreadsGray : kInv4ThreadsRgb;
  dim3 grid((total_pairs + TP - 1) / TP, 1, n);
  const int smem = NCH * 64 * 2 * TP + kInvTableBytes;
  if constexpr (LF == 0) {
    CK(cudaFuncSetAttribute((k_inverse4<NCH, TP>), cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    LAUNCH("k_inverse", (k_inverse4<NCH, TP>), grid, TP, smem, d_planes, d_R, g, d_inv, inv_stride, d_pixels, 1u);
  } else {
    CK(cudaFuncSetAttribute((k_inverse4_scaled<NCH, TP, LF>), cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    LAUNCH("k_inverse4_scaled", (k_inverse4_scaled<NCH, TP, LF>), grid, TP, smem, d_planes, d_R, g, d_inv, inv_stride, d_pixels,
           1u);
  }
  return HIMGCU_OK;
}

// The shapes the lane-pair kernels of a whole-image decode take, for pixel stores store_bytes wide.
bool lane_pair_ok(const himgcu_ctx *ctx, const Geom &g, const uint8_t *d_planes, const uint8_t *d_R, const uint8_t *d_pixels,
                  unsigned store_bytes) {
  return !ctx->force_generic && !(ctx->xform_variant & 1) && (g.h % 8) == 0 && (g.cols % 16) == 0 && (g.w % 16) == 0 &&
         (g.nch == 1 || g.nch == 3) && (reinterpret_cast<uintptr_t>(d_planes) & 15) == 0 &&
         (reinterpret_cast<uintptr_t>(d_pixels) & (store_bytes - 1)) == 0 && (reinterpret_cast<uintptr_t>(d_R) & 1) == 0;
}

// K-inv of a whole-image decode.  lf > 0 (1..3): the decode is scaled by 2^lf, and image i is
// [ceil(h / 2^lf)][ceil(w / 2^lf)][nch] at d_pixels plus i times that size (or at d_pixels + px_off[i] when MIXED).
template <bool MIXED = false>
int stage_inverse(himgcu_ctx *ctx, const uint8_t *d_planes, const uint8_t *d_R, int n, const Geom &g,
                  const DecTables *d_tabs, unsigned long long tab_stride, uint8_t *d_pixels, int lf = 0,
                  const MixedDims &md = {}, const unsigned long long *px_off = nullptr) {
  // lane-pair fast path: two blocks per thread, flat tiles, pixel stores 16 >> lf bytes wide
  if (!MIXED && lane_pair_ok(ctx, g, d_planes, d_R, d_pixels, 16u >> lf)) {
    switch (g.nch * 4 + lf) {
      case 1 * 4 + 0: return launch_inv4<1, 0>(ctx, d_planes, d_R, n, g, d_tabs, tab_stride, d_pixels);
      case 1 * 4 + 1: return launch_inv4<1, 1>(ctx, d_planes, d_R, n, g, d_tabs, tab_stride, d_pixels);
      case 1 * 4 + 2: return launch_inv4<1, 2>(ctx, d_planes, d_R, n, g, d_tabs, tab_stride, d_pixels);
      case 1 * 4 + 3: return launch_inv4<1, 3>(ctx, d_planes, d_R, n, g, d_tabs, tab_stride, d_pixels);
      case 3 * 4 + 0: return launch_inv4<3, 0>(ctx, d_planes, d_R, n, g, d_tabs, tab_stride, d_pixels);
      case 3 * 4 + 1: return launch_inv4<3, 1>(ctx, d_planes, d_R, n, g, d_tabs, tab_stride, d_pixels);
      case 3 * 4 + 2: return launch_inv4<3, 2>(ctx, d_planes, d_R, n, g, d_tabs, tab_stride, d_pixels);
      default: return launch_inv4<3, 3>(ctx, d_planes, d_R, n, g, d_tabs, tab_stride, d_pixels);
    }
  }
  if (!MIXED && !lf && !ctx->force_generic && (g.w % 8) == 0 && (g.h % 8) == 0 && (g.cols % 16) == 0 &&
      (reinterpret_cast<uintptr_t>(d_planes) & 15) == 0 && (reinterpret_cast<uintptr_t>(d_pixels) & 7) == 0 &&
      (((size_t)g.w * g.nch) & 7) == 0) {
    switch (g.nch) {
      case 1: return launch_inv2<1>(ctx, d_planes, d_R, n, g, d_tabs, tab_stride, d_pixels);
      case 3: return launch_inv2<3>(ctx, d_planes, d_R, n, g, d_tabs, tab_stride, d_pixels);
      case 4: return launch_inv2<4>(ctx, d_planes, d_R, n, g, d_tabs, tab_stride, d_pixels);
      default: break;
    }
  }
  return for_channel_groups(g.nch, false, [&](auto nc, int cbase, int ctotal, bool) -> int {
    constexpr int NCH = decltype(nc)::value;
    const dim3 grid((g.cols + kTile - 1) / kTile, g.rows, n);
    if (lf)
      LAUNCH("k_inverse_scaled", (k_inverse_scaled<NCH, MIXED>), grid, kTile, 0, d_planes, d_R, g, d_tabs, tab_stride, d_pixels,
             cbase, ctotal, lf, md, px_off);
    else
      LAUNCH("k_inverse", (k_inverse<NCH, MIXED>), grid, kTile, 0, d_planes, d_R, g, d_tabs, tab_stride, d_pixels, cbase, ctotal,
             md, px_off);
    return HIMGCU_OK;
  });
}

// One Huffman chunk per item, or (image mode) LRES + FRES with the container around them.
struct HuffChunkArgs {
  const uint8_t *d_in;
  HuffGeom hg;
  const char *tag;  // buffer name suffix
  std::vector<uint8_t> prefix;
  int size_patch;
};

// With MIXED the items are the images of a mixed-geometry batch (chunk 0 LRES, chunk 1 FRES, each HuffGeom the
// bounding one; see MixedHuff).  Their chunks have no parts, and force_generic does not apply: the first-generation
// coder has no mixed variant.
template <bool MIXED = false>
int huff_encode_items(himgcu_ctx *ctx, int n, HuffChunkArgs *chunks, int nchunks, bool riff, uint8_t *d_out,
                      size_t out_stride, uint32_t *d_sizes, const MixedDims &md = {}) {
  const bool generic = ctx->force_generic && !MIXED;
  // Device error flag of the encoder (5: code longer than 32 bits, 4: output does not fit, 99: internal
  // mismatch, kEncErrDims: dims out of bounds in a mixed batch).  Sticky per context: cleared when it is read (take_enc_err), not per call, so that an
  // error in an earlier sub-batch of an asynchronous call is not lost.
  int *d_err;
  const bool fresh = ctx->bufs.find("enc_err") == ctx->bufs.end() || ctx->bufs["enc_err"].p == nullptr;
  ENSURE("enc_err", sizeof(int), d_err);
  if (fresh) CK(cudaMemsetAsync(d_err, 0, sizeof(int), ctx->stream));
  LayoutParams P;
  memset(&P, 0, sizeof(P));
  P.nchunks = nchunks;
  P.riff_patch = riff ? 1 : 0;
  P.out = d_out;
  P.out_stride = out_stride;
  P.sizes = d_sizes;
  P.err = d_err;
  // prefixes of all chunks share one small device buffer
  size_t prefix_total = 0;
  for (int k = 0; k < nchunks; ++k) prefix_total += chunks[k].prefix.size();
  uint8_t *d_prefix = nullptr;
  if (prefix_total) {
    ENSURE("enc_prefix", prefix_total, d_prefix);
    std::vector<uint8_t> all;
    for (int k = 0; k < nchunks; ++k) all.insert(all.end(), chunks[k].prefix.begin(), chunks[k].prefix.end());
    const std::string key(all.begin(), all.end());
    if (ctx->prefix_key != key) {
      CK(cudaMemcpyAsync(d_prefix, all.data(), all.size(), cudaMemcpyHostToDevice, ctx->stream));
      CK(cudaStreamSynchronize(ctx->stream));  // `all` is a local
      ctx->prefix_key = key;
    }
  }
  size_t prefix_off = 0;
  TreeOut *d_trees[2];
  uint32_t *d_seghist[2], *d_bits[2], *d_pos[2];
  uint32_t *d_part[2], *d_pbits[2];
  TreeParams TP;
  memset(&TP, 0, sizeof(TP));
  ItemLists lists[2];
  bool teams[2] = {false, false};
  MixedHuff mh[2] = {};  // (the uniform kernels take the default)
  for (int k = 0; k < nchunks; ++k) {
    HuffGeom &hg = chunks[k].hg;
    if (MIXED) mh[k] = MixedHuff{md, k};
    // Parts per segment: only worth it when the segments alone cannot fill the GPU (the low-res chunk
    // of an image is ONE unframed segment: one CTA per image otherwise).  Parts of >= 8 KiB.
    hg.nsub = 1;
    hg.sub_size = hg.seg_size;
    // CTAs wanted: every SM busy for the one-CTA-per-image low-res chunk; framed chunks already have a
    // CTA per block row and only get parts when even those are few (measured: more parts cost more
    // in the layout and look-back steps than they gain)
    const long long ctas = (long long)n * hg.nseg, fill = hg.nseg == 1 ? 148 * 8 : 148 * 2;
    if (!generic && !MIXED && ctas < fill && hg.seg_size > 2 * kTokPiece) {
      const int want = (int)std::min<long long>(64, (fill + ctas - 1) / ctas);
      const int sub = (int)((((long long)hg.seg_size + want - 1) / want + kTokPiece - 1) / kTokPiece) * kTokPiece;
      hg.sub_size = sub;
      hg.nsub = (hg.seg_size + sub - 1) / sub;
    }
    // Warp teams (a warp per segment, eight segments per CTA) for framed chunks whose segments have no parts,
    // when the segments fill every SM with warps: a single 8K image (1024 segments) measured 0.52 ms encode
    // with a CTA per segment, 0.88 ms with a warp per segment.
    const long long wave = 148LL * kTeamWarps * kP4MinCtas;  // resident warps of k_huff_pack4
    teams[k] = !generic && hg.nseg > 1 && hg.nsub == 1 &&
               (ctx->huff_warp_teams == 2 || (ctx->huff_warp_teams == 1 && (long long)n * hg.nseg >= wave));
    const std::string tag = chunks[k].tag;
    ENSURE((tag + "_seghist").c_str(), (size_t)n * hg.nseg * hg.nsub * kSyms * sizeof(uint32_t), d_seghist[k]);
    ENSURE((tag + "_partstart").c_str(), (size_t)n * hg.nseg * hg.nsub * sizeof(uint32_t), d_part[k]);
    ENSURE((tag + "_trees").c_str(), (size_t)n * sizeof(TreeOut), d_trees[k]);
    ENSURE((tag + "_segbits").c_str(), (size_t)n * hg.nseg * sizeof(uint32_t), d_bits[k]);
    ENSURE((tag + "_segpos").c_str(), (size_t)n * hg.nseg * sizeof(uint32_t), d_pos[k]);
    dim3 grid(hg.nseg * hg.nsub, n);
    // item lists of the pieces, handed from the histogram pass to the packer (see ItemLists)
    ItemLists &il = lists[k];
    il = ItemLists{nullptr, nullptr, nullptr, 0};
    if (!generic && ctx->item_lists) {
      const int ppp = (hg.sub_size + kTokPiece - 1) / kTokPiece;
      const size_t slots = (size_t)n * hg.nseg * hg.nsub * ppp;
      ENSURE((tag + "_itpos").c_str(), slots * kItemCap * sizeof(unsigned short), il.pos);
      ENSURE((tag + "_itval").c_str(), slots * kItemCap, il.val);
      ENSURE((tag + "_itcnt").c_str(), slots * sizeof(uint32_t), il.count);
      il.pieces_per_part = ppp;
    }
    ENSURE((tag + "_partbits").c_str(), (size_t)n * hg.nseg * hg.nsub * sizeof(uint32_t), d_pbits[k]);
    uint32_t *d_total = nullptr;
    if (!generic) {  // chunk histograms summed by the histogram kernel itself
      ENSURE((tag + "_histtotal").c_str(), (size_t)n * kSyms * sizeof(uint32_t), d_total);
      CK(cudaMemsetAsync(d_total, 0, (size_t)n * kSyms * sizeof(uint32_t), ctx->stream));
    }
    const dim3 team_grid((hg.nseg + kTeamWarps - 1) / kTeamWarps, n);
    if (generic) LAUNCH("k_huff_hist", k_huff_hist, grid, kHuffThreads, 0, chunks[k].d_in, hg, d_seghist[k]);
    else if (teams[k])
      LAUNCH("k_huff_hist", k_huff_hist4<MIXED>, team_grid, kTeamThreads, 0, chunks[k].d_in, hg, d_seghist[k], il, d_total, mh[k]);
    else LAUNCH("k_huff_hist", k_huff_hist2<MIXED>, grid, kTokThreads, 0, chunks[k].d_in, hg, d_seghist[k], il, d_total, mh[k]);
    TP.total[k] = d_total;
    TP.seghist[k] = d_seghist[k];
    TP.trees[k] = d_trees[k];
    TP.rows[k] = hg.nseg * hg.nsub;
    LayoutChunk &C = P.ch[k];
    C.part_bits = d_pbits[k];
    C.seghist = d_seghist[k];
    C.trees = d_trees[k];
    C.seg_bits = d_bits[k];
    C.seg_pos = d_pos[k];
    C.part_start = d_part[k];
    C.nsub = hg.nsub;
    C.prefix = chunks[k].prefix.empty() ? nullptr : d_prefix + prefix_off;
    C.prefix_len = (int)chunks[k].prefix.size();
    C.size_patch = chunks[k].size_patch;
    C.nseg = hg.nseg;
    C.framed = hg.nseg > 1 ? 1 : 0;
    prefix_off += chunks[k].prefix.size();
  }
  LAUNCH("k_huff_tree", k_huff_tree, dim3(n, nchunks), kTreeThreads, 0, TP, d_err);
  for (int k = 0; k < nchunks; ++k) {
    const int rows = chunks[k].hg.nseg * chunks[k].hg.nsub;
    LAUNCH("k_huff_layout", k_huff_segbits, dim3((rows + 7) / 8, n), 256, 0, d_seghist[k], d_trees[k], rows, d_pbits[k]);
  }
  if (MIXED) LAUNCH("k_huff_layout", k_huff_layout_mixed, n, kLayoutThreads, 0, P, md, ContainerTemplate::kDimsAt);
  else LAUNCH("k_huff_layout", k_huff_layout, n, kLayoutThreads, 0, P);
  const size_t win_bytes = (kWinWords + 2) * sizeof(uint32_t);
  if (generic)  // static + dynamic shared memory of the first-generation packer exceed 48 KiB
    CK(cudaFuncSetAttribute(k_huff_pack, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)win_bytes));
  if (teams[0] || teams[1]) CK(cudaFuncSetAttribute(k_huff_pack4<MIXED>, cudaFuncAttributeMaxDynamicSharedMemorySize, kP4Smem));
  for (int k = 0; k < nchunks; ++k) {
    const HuffGeom &hg = chunks[k].hg;
    dim3 grid(hg.nseg * hg.nsub, n);
    if (generic)
      LAUNCH("k_huff_pack", k_huff_pack, grid, kHuffThreads, win_bytes, chunks[k].d_in, hg, d_trees[k], d_bits[k],
             d_pos[k], d_sizes, d_out, (unsigned long long)out_stride, d_err);
    else if (teams[k])
      LAUNCH("k_huff_pack", k_huff_pack4<MIXED>, dim3((hg.nseg + kTeamWarps - 1) / kTeamWarps, n), kTeamThreads, kP4Smem,
             chunks[k].d_in, hg, d_trees[k], d_bits[k], d_pos[k], d_sizes, d_out, (unsigned long long)out_stride, d_err, lists[k],
             mh[k]);
    else
      LAUNCH("k_huff_pack", k_huff_pack3<MIXED>, grid, kTokThreads, 0, chunks[k].d_in, hg, d_trees[k], d_bits[k], d_pos[k],
             d_part[k], d_sizes, d_out, (unsigned long long)out_stride, d_err, lists[k], mh[k]);
    if (hg.nseg > 1)
      LAUNCH("k_huff_stale", k_huff_stale<MIXED>, dim3((hg.nseg + 255) / 256, n), 256, 0, n, hg.nseg, d_bits[k], d_pos[k], d_sizes,
             d_out, (unsigned long long)out_stride, md);
  }
  return HIMGCU_OK;
}
// Instantiated here, before the stages that encode_device calls ahead of it: the module's extern shared arrays are
// declared in instantiation order, and where k_forward3's 128-byte aligned one comes before k_huff_pack4's 16-byte
// aligned window, ptxas starts that window 80 bytes later (0x880 instead of 0x830) and allocates k_huff_pack4's
// registers differently.
template int huff_encode_items<false>(himgcu_ctx *, int, HuffChunkArgs *, int, bool, uint8_t *, size_t, uint32_t *,
                                      const MixedDims &);
template int huff_encode_items<true>(himgcu_ctx *, int, HuffChunkArgs *, int, bool, uint8_t *, size_t, uint32_t *,
                                     const MixedDims &);

int read_err_flag(himgcu_ctx *ctx, const char *name, int *value) {
  int *d_err;
  ENSURE(name, sizeof(int), d_err);
  CK(cudaMemcpyAsync(value, d_err, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemsetAsync(d_err, 0, sizeof(int), ctx->stream));  // read = clear
  CK(cudaStreamSynchronize(ctx->stream));
  return HIMGCU_OK;
}

// Status code of a device encoder error flag value (0 = none).
int enc_err_status(himgcu_ctx *ctx, int err) {
  if (err == 5) return fail(ctx, HIMGCU_ERR_UNSUPPORTED, "Huffman code longer than 32 bits");
  if (err == 99) return fail(ctx, HIMGCU_ERR_CUDA, "internal: packed size mismatch");
  if (err == kEncErrDims) return fail(ctx, HIMGCU_ERR_ARG, "image dims below 1 or above the bounds");
  if (err) return fail(ctx, HIMGCU_ERR_CAPACITY, "internal output bound exceeded");
  return HIMGCU_OK;
}

size_t per_image_encode_ws(const Geom &g) {
  return 2 * (size_t)g.nch * g.rows * g.cols + g.lres_stride + g.planes_bytes +
         (size_t)(g.rows + 1) * kSyms * 4 + 2 * sizeof(TreeOut) + (size_t)(g.rows + 1) * 8 +
         // item lists: 3 bytes x kItemCap per 8 KiB piece of the planes and of the low-res chunk
         ((size_t)g.rows * ((g.seg + kTokPiece - 1) / kTokPiece) + (g.lres_size + kTokPiece - 1) / kTokPiece + 64) *
             (kItemCap * 3 + 4);
}

// Whole-image encode of a sub-batch already resident on the device.
template <bool MIXED = false>
int encode_device(himgcu_ctx *ctx, const uint8_t *d_pixels, int n, const Geom &g, int quality, bool ycbcr,
                  uint8_t *d_out, size_t out_stride, uint32_t *d_sizes, const MixedDims &md = {},
                  const unsigned long long *px_off = nullptr) {
  EncodeTables t;
  BuildEncodeTables(quality, ycbcr, &t);
  ContainerTemplate ct;
  BuildContainerTemplate(t, g.w, g.h, g.nch, &ct);
  uint8_t *d_L, *d_lres, *d_planes;
  ENSURE("L", (size_t)n * g.nch * g.rows * g.cols, d_L);
  ENSURE("lres", (size_t)n * g.lres_stride, d_lres);
  ENSURE("planes", (size_t)n * g.planes_bytes, d_planes);
  int rc = stage_lowres<MIXED>(ctx, d_pixels, n, g, ycbcr, d_L, md, px_off);
  if (rc) return rc;
  rc = stage_lres_encode<MIXED>(ctx, d_L, n, g, t, d_lres, md);
  if (rc) return rc;
  rc = stage_forward<MIXED>(ctx, d_pixels, d_L, n, g, t, d_planes, md, px_off);
  if (rc) return rc;
  HuffChunkArgs ch[2];
  ch[0].d_in = d_lres;
  ch[0].hg = HuffGeom{g.lres_size, 1, g.lres_stride, 1, g.lres_size};
  ch[0].tag = "lres";
  ch[0].prefix = ct.head;
  ch[0].size_patch = (int)ct.head.size() - 4;
  ch[1].d_in = d_planes;
  ch[1].hg = HuffGeom{g.seg, g.rows, g.planes_bytes, 1, g.seg};
  ch[1].tag = "fres";
  ch[1].prefix = ct.mid;
  ch[1].size_patch = (int)ct.mid.size() - 4;
  return huff_encode_items<MIXED>(ctx, n, ch, 2, true, d_out, out_stride, d_sizes, md);
}

// Threads per stream for k_dec_stream_par: grow the team until ~128k threads are in flight, but keep
// at least ~256 output bytes per thread.
int decode_team(long long streams, int out_bytes, int base) {
  int team = base;
  while (team < kParMaxTeam && streams * team < 131072 && out_bytes / (team * 2) >= 256) team *= 2;
  return team;
}

// One unframed stream per item, decoded by a thread-block cluster of kDecCluster CTAs (distributed
// shared memory) when there are few, large streams: a single image's low-res chunk.
constexpr int kDecCluster = 8;
bool use_decode_cluster(long long streams, int out_bytes) { return streams <= 16 && out_bytes >= (64 << 10); }
int launch_stream_cluster(himgcu_ctx *ctx, const char *name, int n, const uint8_t *d_in, const ChunkDesc *d_cd,
                          const DecTree *d_tree, const SegRef *d_seg, int out_seg, uint8_t *d_out,
                          unsigned long long out_stride, int *d_status, bool *launched) {
  // Not the widest team possible: where the stream is periodic (flat areas repeat one code) wrongly
  // started decoders never re-synchronise and the rounds advance one subsequence at a time, so very
  // short subsequences cost more rounds than they save work (measured on 4K and 8K images).
  const int threads = out_seg >= (256 << 10) ? 512 : 256;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(kDecCluster, n);
  cfg.blockDim = dim3(threads);
  cfg.stream = ctx->stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = kDecCluster;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  // a cluster of 8 CTAs must be co-schedulable (it is on a whole B200; not necessarily on a partitioned
  // one): ask first, and let the caller fall back to the one-CTA team otherwise
  int max_clusters = 0;
  if (cudaOccupancyMaxActiveClusters(&max_clusters, k_dec_stream_par<false, kDecCluster>, &cfg) != cudaSuccess || max_clusters < 1) {
    cudaGetLastError();
    *launched = false;
    return HIMGCU_OK;
  }
  cudaError_t e;
  {
    LaunchScope ls_(ctx, name);
    e = cudaLaunchKernelEx(&cfg, k_dec_stream_par<false, kDecCluster>, d_in, d_cd, d_tree, const_cast<SegRef *>(d_seg), 1, out_seg,
                           d_out, out_stride, d_status, 0, 0, MixedDims{});
  }
  if (e != cudaSuccess) return fail(ctx, HIMGCU_ERR_CUDA, "launch %s failed: %s", name, cudaGetErrorString(e));
  *launched = true;
  return HIMGCU_OK;
}

// nseg framed segments per item from a segment table: a warp per segment (kParWarpTeams per CTA) when team == 32,
// otherwise a CTA of `team` threads per segment.  MIX: the mixed-geometry mode of k_dec_stream_par (0 = uniform).
template <int MIX = 0>
int launch_stream_segments(himgcu_ctx *ctx, const char *name, int team, int n, const uint8_t *d_in, const ChunkDesc *d_cd,
                           const DecTree *d_tree, SegRef *d_seg, int nseg, int out_seg, uint8_t *d_out,
                           unsigned long long out_stride, int *d_status, const MixedDims &md = {}) {
  if (team == 32)
    LAUNCH(name, (k_dec_stream_par<true, 1, MIX>), dim3((nseg + kParWarpTeams - 1) / kParWarpTeams, n), 32 * kParWarpTeams, 0,
           d_in, d_cd, d_tree, d_seg, nseg, out_seg, d_out, out_stride, d_status, 0, 0, md);
  else
    LAUNCH(name, (k_dec_stream_par<false, 1, MIX>), dim3(nseg, n), team, 0, d_in, d_cd, d_tree, d_seg, nseg, out_seg, d_out,
           out_stride, d_status, 0, 0, md);
  return HIMGCU_OK;
}

// Device scratch of a decode (whole image or region) that decode_front fills.
struct DecFront {
  const ChunkDesc *fcd;
  const DecTree *ftree;
  const DecTables *tabs;
  SegRef *fseg;  // [n][rows]
  uint8_t *R;    // decoded low-res images
  bool fork;     // the low-res branch runs on ctx->aux_stream: wait for ctx->ev_join before reading R
};

// What every decode does before the coefficient planes: container, tables and both trees of n streams, then
// the low-res branch (segment table, stream, DPCM into R).  The caller ensures its planes buffer before: a
// workspace that grows is freed after a stream synchronisation, which must not happen while the two branches
// of a single image run on two streams.  With MIXED the low-res stream of an image is never given to a cluster.
template <bool MIXED = false>
int decode_front(himgcu_ctx *ctx, const uint8_t *d_himg, const unsigned long long *d_offsets, const uint32_t *d_sizes, int n,
                 const Geom &g, int lenient, int *d_status, DecFront *f, const MixedDims &md = {}) {
  ChunkDesc *d_lcd, *d_fcd;
  DecTables *d_tabs;
  DecTree *d_ltree, *d_ftree;
  SegRef *d_lseg, *d_fseg;
  uint8_t *d_lres, *d_R;
  ENSURE("dec_lcd", (size_t)n * sizeof(ChunkDesc), d_lcd);
  ENSURE("dec_fcd", (size_t)n * sizeof(ChunkDesc), d_fcd);
  ENSURE("dec_tabs", (size_t)n * sizeof(DecTables), d_tabs);
  ENSURE("dec_ltree", (size_t)n * sizeof(DecTree), d_ltree);
  ENSURE("dec_ftree", (size_t)n * sizeof(DecTree), d_ftree);
  ENSURE("dec_lseg", (size_t)n * sizeof(SegRef), d_lseg);
  ENSURE("dec_fseg", (size_t)n * g.rows * sizeof(SegRef), d_fseg);
  ENSURE("lres", (size_t)n * g.lres_stride, d_lres);
  ENSURE("L", (size_t)n * g.nch * g.rows * g.cols, d_R);
  *f = DecFront{d_fcd, d_ftree, d_tabs, d_fseg, d_R, n == 1 && !ctx->profile};
  const unsigned nb = (unsigned)((n + 127) / 128);
  LAUNCH("k_dec_parse", k_dec_parse<MIXED>, (unsigned)((n + 3) / 4), 128, 0, d_himg, d_offsets, d_sizes, n, g.w, g.h, g.nch, d_lcd,
         d_fcd, d_tabs, d_status, md);
  LAUNCH("k_dec_tree", k_dec_tree, dim3(n, 2), kDecTreeThreads, 0, d_himg, d_lcd, d_fcd, lenient, d_ltree, d_ftree, d_status);
  // A single image is a chain of latency-bound kernels: its two branches (low-res stream -> DPCM, and
  // segment table -> coefficient planes) share nothing until the inverse transform, so they run on
  // two streams.  Batches fill the GPU on one stream (and device-side event waits are kept out of
  // the multi-context host pipelines, see run_pipeline).
  const bool fork = f->fork;
  cudaStream_t main_stream = ctx->stream;
  if (fork) {
    if (!ctx->aux_stream) {
      CK(cudaStreamCreateWithFlags(&ctx->aux_stream, cudaStreamNonBlocking));
      CK(cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
      CK(cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming));
    }
    CK(cudaEventRecord(ctx->ev_fork, main_stream));
    CK(cudaStreamWaitEvent(ctx->aux_stream, ctx->ev_fork, 0));
    ctx->stream = ctx->aux_stream;  // the LAUNCH macro launches on ctx->stream
  }
  auto lres_branch = [&]() -> int {
    LAUNCH("k_dec_segtab", k_dec_segtab, nb, 128, 0, d_himg, d_lcd, d_ltree, n, 1, g.lres_size, 0, lenient, d_lseg,
           d_status);
    // one CTA per stream.  Team size: 256 threads per LRES stream when the batch alone fills the GPU,
    // wider teams (or a cluster of CTAs) when there are few streams (single images).
    const int lres_team = decode_team(n, g.lres_size, kParLresThreads);
    bool clustered = false;
    if (!MIXED && use_decode_cluster(n, g.lres_size) && !ctx->force_generic) {
      int rc = launch_stream_cluster(ctx, "k_dec_stream_lres", n, d_himg, d_lcd, d_ltree, d_lseg, g.lres_size, d_lres,
                                     (unsigned long long)g.lres_stride, d_status, &clustered);
      if (rc) return rc;
    }
    if (!clustered)
      LAUNCH("k_dec_stream_lres", (k_dec_stream_par<false, 1, MIXED ? kMixLres : 0>), dim3(1, n), lres_team, 0, d_himg, d_lcd,
             d_ltree, d_lseg, 1, g.lres_size, d_lres, g.lres_stride, d_status, 0, 0, md);
    const long long nmb = (long long)n * g.nch * g.mrows * g.mcols;
    const unsigned blocks = (unsigned)((nmb + kLresWarps * 2 - 1) / (kLresWarps * 2));
    LAUNCH("k_lres_dpcm_dec", (k_lres_dpcm<false, MIXED>), blocks, kLresWarps * 32, 0, (const uint8_t *)nullptr, d_lres, d_R, g, n,
           (const uint8_t *)nullptr, d_tabs->low_unmap, (unsigned long long)sizeof(DecTables), md);
    return HIMGCU_OK;
  };
  int rc_l = lres_branch();
  ctx->stream = main_stream;
  if (fork) {  // (also when the branch failed: its work must be ordered before the next call on the main stream)
    CK(cudaEventRecord(ctx->ev_join, ctx->aux_stream));
    if (rc_l) CK(cudaStreamWaitEvent(main_stream, ctx->ev_join, 0));
  }
  return rc_l;
}

// Whole-image decode of n streams resident on the device.  lf > 0: every image is written scaled by 2^lf (see
// stage_inverse); everything before the inverse transform is the same.
template <bool MIXED = false>
int decode_device(himgcu_ctx *ctx, const uint8_t *d_himg, const unsigned long long *d_offsets, const uint32_t *d_sizes, int n,
                  const Geom &g, int flags, uint8_t *d_pixels, int *d_status, int lf = 0, const MixedDims &md = {},
                  const unsigned long long *px_off = nullptr) {
  const int lenient = (flags & HIMGCU_LENIENT) ? 1 : 0;
  uint8_t *d_planes;
  ENSURE("planes", (size_t)n * g.planes_bytes, d_planes);
  DecFront f;
  int rc = decode_front<MIXED>(ctx, d_himg, d_offsets, d_sizes, n, g, lenient, d_status, &f, md);
  if (rc) return rc;
  // a warp per block row when the batch alone fills the GPU, wider teams for few streams
  const int fres_team = decode_team((long long)n * g.rows, g.seg, kParFresThreads);
  // Few streams (single images): the serial walk over the segment headers runs inside the decode kernel
  // and the rows decode as soon as their entry is published (all CTAs of such a grid are resident at once).
  // A mixed batch has no inline walk; block rows past an image's own are idle in its stream decoder.
  const bool inline_walk =
      !MIXED && fres_team > 32 && !ctx->force_generic && (long long)n * (g.rows + 1) * fres_team <= 148LL * 2048;
  if (inline_walk) {
    CK(cudaMemsetAsync(f.fseg, 0xfe, (size_t)n * g.rows * sizeof(SegRef), ctx->stream));  // kSegNotReady
    LAUNCH("k_dec_stream_fres", k_dec_stream_par<false>, dim3(g.rows + 1, n), fres_team, 0, d_himg, f.fcd, f.ftree, f.fseg,
           g.rows, g.seg, d_planes, g.planes_bytes, d_status, 1, lenient);
  } else {
    const unsigned nb = (unsigned)((n + 127) / 128);
    if (MIXED)
      LAUNCH("k_dec_segtab", k_dec_segtab_mixed, nb, 128, 0, d_himg, f.fcd, f.ftree, n, g.rows, lenient, f.fseg, d_status, md);
    else
      LAUNCH("k_dec_segtab", k_dec_segtab, nb, 128, 0, d_himg, f.fcd, f.ftree, n, g.rows, g.seg, 1, lenient, f.fseg, d_status);
    rc = launch_stream_segments<MIXED ? kMixWhole : 0>(ctx, "k_dec_stream_fres", fres_team, n, d_himg, f.fcd, f.ftree, f.fseg,
                                                        g.rows, g.seg, d_planes, g.planes_bytes, d_status, md);
    if (rc) return rc;
  }
  if (f.fork) CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_join, 0));
  return stage_inverse<MIXED>(ctx, d_planes, f.R, n, g, f.tabs, sizeof(DecTables), d_pixels, lf, md, px_off);
}

// Compact block rows a region decode keeps per image: the most a rectangle of rh rows can touch.  Scaled by 2^lf, the
// rectangle reads at most (rh << lf) source rows from a row that is a multiple of 2^lf.
int region_rows(const Geom &g, int rh, int lf = 0) { return std::min(((rh << lf) + 15 - (1 << lf)) / 8, g.rows); }

// Lane-pair inverse of a region decode scaled by 2^LF (LF in 1..3): k_inverse_region4_scaled.
template <int NCH, int LF>
int launch_inv_region4_scaled(himgcu_ctx *ctx, const uint8_t *d_planes, const uint8_t *d_R, int n, const Geom &g,
                              const InvTables *d_inv, const int32_t *d_origins, int rw, int rh, int kr, uint8_t *d_pixels) {
  constexpr int TP = kInv4ThreadsRgb;
  const int span = region_span_pairs(rw << LF, g.cols);
  dim3 grid((unsigned)(((long long)kr * span + TP - 1) / TP), 1, n);
  const int smem = NCH * 64 * 2 * TP + kInvTableBytes;
  CK(cudaFuncSetAttribute((k_inverse_region4_scaled<NCH, TP, LF>), cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  LAUNCH("k_inverse_region4_scaled", (k_inverse_region4_scaled<NCH, TP, LF>), grid, TP, smem, d_planes, d_R, g, d_inv,
         (unsigned long long)sizeof(InvTables), d_origins, rw, rh, kr, span, d_pixels, 1u);
  return HIMGCU_OK;
}

// K-inv of a region decode (xform_region.cuh) from the compact planes [n][kr][seg].  lf > 0 (1..3): the rectangle is
// one of the image scaled by 2^lf.
template <bool MIXED = false>
int stage_inverse_region(himgcu_ctx *ctx, const uint8_t *d_planes, const uint8_t *d_R, int n, const Geom &g,
                         const DecTables *d_tabs, const int32_t *d_origins, int rw, int rh, int kr, uint8_t *d_pixels,
                         const MixedDims &md = {}, int lf = 0) {
  if (lf) {
    // lane-pair fast path: the shapes k_inverse4_scaled takes (every window whole), the rectangle clips rows and columns
    // (the clipped stores take any output alignment)
    if (!MIXED && lane_pair_ok(ctx, g, d_planes, d_R, d_pixels, 1u)) {
      InvTables *d_inv;
      int rc = launch_inv_tables(ctx, d_tabs, n, (unsigned long long)sizeof(DecTables), &d_inv);
      if (rc) return rc;
      switch (g.nch * 4 + lf) {
        case 1 * 4 + 1: return launch_inv_region4_scaled<1, 1>(ctx, d_planes, d_R, n, g, d_inv, d_origins, rw, rh, kr, d_pixels);
        case 1 * 4 + 2: return launch_inv_region4_scaled<1, 2>(ctx, d_planes, d_R, n, g, d_inv, d_origins, rw, rh, kr, d_pixels);
        case 1 * 4 + 3: return launch_inv_region4_scaled<1, 3>(ctx, d_planes, d_R, n, g, d_inv, d_origins, rw, rh, kr, d_pixels);
        case 3 * 4 + 1: return launch_inv_region4_scaled<3, 1>(ctx, d_planes, d_R, n, g, d_inv, d_origins, rw, rh, kr, d_pixels);
        case 3 * 4 + 2: return launch_inv_region4_scaled<3, 2>(ctx, d_planes, d_R, n, g, d_inv, d_origins, rw, rh, kr, d_pixels);
        default: return launch_inv_region4_scaled<3, 3>(ctx, d_planes, d_R, n, g, d_inv, d_origins, rw, rh, kr, d_pixels);
      }
    }
    const int kb = ((rw << lf) + 15 - (1 << lf)) / 8;
    LAUNCH("k_inverse_region_scaled", k_inverse_region_scaled<MIXED>, dim3((kb + kTile - 1) / kTile, kr, n), kTile, 0, d_planes, d_R,
           g, d_tabs, (unsigned long long)sizeof(DecTables), d_origins, rw, rh, kr, lf, d_pixels, md);
    return HIMGCU_OK;
  }
  // lane-pair fast path: the shapes k_inverse4 takes, except that the rectangle clips rows and columns
  if (!MIXED && !ctx->force_generic && (g.cols % 16) == 0 && (g.nch == 1 || g.nch == 3) &&
      (reinterpret_cast<uintptr_t>(d_planes) & 15) == 0 && (reinterpret_cast<uintptr_t>(d_R) & 1) == 0) {
    InvTables *d_inv;
    int rc = launch_inv_tables(ctx, d_tabs, n, (unsigned long long)sizeof(DecTables), &d_inv);
    if (rc) return rc;
    const int span = region_span_pairs(rw, g.cols);
    constexpr int TP = kInv4ThreadsRgb;
    static_assert(kInv4ThreadsGray == TP, "one tile width for both channel counts");
    dim3 grid((unsigned)(((long long)kr * span + TP - 1) / TP), 1, n);
    const int smem = g.nch * 64 * 2 * TP + kInvTableBytes;
    if (g.nch == 1) {
      CK(cudaFuncSetAttribute((k_inverse_region4<1, TP>), cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
      LAUNCH("k_inverse_region4", (k_inverse_region4<1, TP>), grid, TP, smem, d_planes, d_R, g, d_inv,
             (unsigned long long)sizeof(InvTables), d_origins, rw, rh, kr, span, d_pixels, 1u);
    } else {
      CK(cudaFuncSetAttribute((k_inverse_region4<3, TP>), cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
      LAUNCH("k_inverse_region4", (k_inverse_region4<3, TP>), grid, TP, smem, d_planes, d_R, g, d_inv,
             (unsigned long long)sizeof(InvTables), d_origins, rw, rh, kr, span, d_pixels, 1u);
    }
    return HIMGCU_OK;
  }
  const int kb = (rw + 14) / 8;
  LAUNCH("k_inverse_region", k_inverse_region<MIXED>, dim3((kb + kTile - 1) / kTile, kr, n), kTile, 0, d_planes, d_R, g, d_tabs,
         (unsigned long long)sizeof(DecTables), d_origins, rw, rh, kr, d_pixels, md);
  return HIMGCU_OK;
}

// Region decode of n streams resident on the device: image i's rectangle rw x rh at (d_origins[2i], d_origins[2i+1])
// to d_pixels + i * rw * rh * nch.  Only the FRES segments of the block rows the rectangle touches are decoded.
// lf > 0: the rectangle is one of the image scaled by 2^lf, and the rows are those of the source pixels it reads.
template <bool MIXED = false>
int decode_region_device(himgcu_ctx *ctx, const uint8_t *d_himg, const unsigned long long *d_offsets, const uint32_t *d_sizes,
                         int n, const Geom &g, int flags, const int32_t *d_origins, int rw, int rh, uint8_t *d_pixels,
                         int *d_status, const MixedDims &md = {}, int lf = 0) {
  const int lenient = (flags & HIMGCU_LENIENT) ? 1 : 0;
  const int kr = region_rows(g, rh, lf);
  uint8_t *d_planes;
  SegRef *d_rseg;
  ENSURE("planes", (size_t)n * kr * g.seg, d_planes);
  ENSURE("dec_rseg", (size_t)n * kr * sizeof(SegRef), d_rseg);
  DecFront f;
  int rc = decode_front<MIXED>(ctx, d_himg, d_offsets, d_sizes, n, g, lenient, d_status, &f, md);
  if (rc) return rc;
  if (lf)
    LAUNCH("k_dec_segtab_region", k_dec_segtab_region_scaled<MIXED>, (unsigned)((n + 127) / 128), 128, 0, d_himg, f.fcd, f.ftree,
           n, g, lenient, d_origins, rw, rh, kr, lf, f.fseg, d_rseg, d_status, md);
  else
    LAUNCH("k_dec_segtab_region", k_dec_segtab_region<MIXED>, (unsigned)((n + 127) / 128), 128, 0, d_himg, f.fcd, f.ftree, n, g,
           lenient, d_origins, rw, rh, kr, f.fseg, d_rseg, d_status, md);
  const int team = decode_team((long long)n * kr, g.seg, kParFresThreads);
  rc = launch_stream_segments<MIXED ? kMixFres : 0>(ctx, "k_dec_stream_fres", team, n, d_himg, f.fcd, f.ftree, d_rseg, kr, g.seg,
                                                     d_planes, (unsigned long long)kr * g.seg, d_status, md);
  if (rc) return rc;
  if (f.fork) CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_join, 0));
  return stage_inverse_region<MIXED>(ctx, d_planes, f.R, n, g, f.tabs, d_origins, rw, rh, kr, d_pixels, md, lf);
}

// Runs body(i0, m) over the sub-batches [i0, i0 + m) of n images: as many images as fit max_workspace_bytes at `per`
// workspace bytes each, at least one and at most 65535.
template <class F>
int for_sub_batches(himgcu_ctx *ctx, int n, size_t per, F &&body) {
  int sub = (int)std::min<size_t>((size_t)n, std::max<size_t>(1, ctx->max_workspace / per));
  sub = std::min(sub, 65535);
  for (int i0 = 0; i0 < n; i0 += sub) {
    const int rc = body(i0, std::min(sub, n - i0));
    if (rc) return rc;
  }
  return HIMGCU_OK;
}

}  // namespace
extern "C" int himgcu_create(int device, himgcu_ctx **out);
extern "C" void himgcu_destroy(himgcu_ctx *ctx);
namespace {

// One copy queue per direction and device, shared by every context of the process: transfers of
// concurrent contexts (say one encoding, one decoding) then run in issue order.  A copy engine keeps
// serving the stream that keeps feeding it: with separate streams a one-megabyte copy of one call was
// measured to wait 30 ms until the other call's stream of 100 MB copies had drained (and for the same
// reason NO copy may be issued on a coding lane's own stream, see the size read-back of the encoder).
struct CopyQueues {
  cudaStream_t in = nullptr, out = nullptr;
};
std::mutex g_copyq_mutex;
std::map<int, CopyQueues> g_copyq;

int ensure_pipeline(himgcu_ctx *ctx) {
  if (ctx->in_stream) return HIMGCU_OK;
  {
    std::lock_guard<std::mutex> lock(g_copyq_mutex);
    CopyQueues &q = g_copyq[ctx->device];
    if (!q.in) {
      CK(cudaStreamCreateWithFlags(&q.in, cudaStreamNonBlocking));
      CK(cudaStreamCreateWithFlags(&q.out, cudaStreamNonBlocking));
    }
    ctx->in_stream = q.in;
    ctx->out_stream = q.out;
  }
  for (int b = 0; b < himgcu_ctx::kMaxLanes; ++b) {
    CK(cudaEventCreateWithFlags(&ctx->ev_in[b], cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&ctx->ev_cmp[b], cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&ctx->ev_out[b], cudaEventDisableTiming));
  }
  return HIMGCU_OK;
}

int ensure_pinned(himgcu_ctx *ctx, size_t bytes) {
  if (ctx->pinned_cap >= bytes) return HIMGCU_OK;
  if (ctx->pinned) {
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaFreeHost(ctx->pinned));
    ctx->pinned = nullptr;
    ctx->pinned_cap = 0;
  }
  CK(cudaMallocHost(&ctx->pinned, bytes));
  ctx->pinned_cap = bytes;
  return HIMGCU_OK;
}

// HIMG_DEBUG_PIPE=1: device-side timeline of the host-buffer calls (ms since the first traced call of
// the process; one line per sub-batch) on stderr.  Debug aid only.
struct PipeTrace {
  bool on = getenv("HIMG_DEBUG_PIPE") != nullptr;
  const char *tag;
  std::vector<cudaEvent_t> ev;  // 4 per sub-batch: copy-in start / end, coding end, copy-out end
  std::vector<double> host;     // host clock when the coding of the sub-batch was launched
  static double now() {
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
  }
  static double &host_epoch() {
    static double t = 0;
    return t;
  }
  static cudaEvent_t epoch() {
    static cudaEvent_t e = [] {
      cudaEvent_t x;
      cudaEventCreate(&x);
      cudaEventRecord(x, 0);
      cudaEventSynchronize(x);
      host_epoch() = now();
      return x;
    }();
    return e;
  }
  void launched(int k) {
    if (!on) return;
    if ((int)host.size() <= k) host.resize(k + 1, 0);
    host[k] = now() - host_epoch();
  }
  explicit PipeTrace(const char *t) : tag(t) {
    if (on) epoch();
  }
  void mark(int k, int what, cudaStream_t s) {
    if (!on) return;
    if ((int)ev.size() < 4 * (k + 1)) ev.resize(4 * (k + 1), nullptr);
    cudaEventCreate(&ev[4 * k + what]);
    cudaEventRecord(ev[4 * k + what], s);
  }
  ~PipeTrace() {
    if (!on) return;
    for (size_t k = 0; k * 4 < ev.size(); ++k) {
      float t[4] = {-1, -1, -1, -1};
      for (int j = 0; j < 4; ++j)
        if (ev[4 * k + j]) {
          cudaEventSynchronize(ev[4 * k + j]);
          cudaEventElapsedTime(&t[j], epoch(), ev[4 * k + j]);
          cudaEventDestroy(ev[4 * k + j]);
        }
      fprintf(stderr, "[pipe %s] sub %2zu  in %8.2f..%8.2f  coded %8.2f  out %8.2f  (launched by the host at %8.2f)\n", tag, k,
              t[0], t[1], t[2], t[3], k < host.size() ? host[k] : -1.0);
    }
  }
};

// Lanes in use for a host-buffer call of K sub-batches; creates the child contexts on demand.
int prepare_lanes(himgcu_ctx *ctx, int K, int *count) {
  int S = std::max(1, std::min({ctx->host_lanes, (int)himgcu_ctx::kMaxLanes, K}));
  if (ctx->profile) S = 1;  // per-kernel events are only meaningful without overlap
  while ((int)ctx->lanes.size() < S - 1) {
    himgcu_ctx *l = nullptr;
    if (himgcu_create(ctx->device, &l) != HIMGCU_OK) return fail(ctx, HIMGCU_ERR_CUDA, "cannot create a coding lane");
    ctx->lanes.push_back(l);
  }
  for (himgcu_ctx *l : ctx->lanes) {
    l->force_generic = ctx->force_generic;
    l->item_lists = ctx->item_lists;
    l->huff_warp_teams = ctx->huff_warp_teams;
    l->max_workspace = ctx->max_workspace;
  }
  *count = S;
  return HIMGCU_OK;
}
himgcu_ctx *lane_of(himgcu_ctx *ctx, int b) { return b == 0 ? ctx : ctx->lanes[b - 1]; }

int finish_lanes(himgcu_ctx *ctx, int S) {
  for (int b = 0; b < S; ++b) CK(cudaStreamSynchronize(lane_of(ctx, b)->stream));
  for (himgcu_ctx *l : ctx->lanes) {
    ctx->launches += l->launches;
    l->launches = 0;
  }
  return HIMGCU_OK;
}

// Host-buffer batches are pipelined: sub-batches flow through the H2D queue, a coding lane and the
// D2H queue, S of them in flight (S device staging slots, S lanes).  The calling thread drives the
// pipeline and orders the stages ON THE HOST (event queries): no stream ever waits on an event of
// another stream.  Device-side waits looked cheaper but a stream parked on one was observed to
// starve for the whole call while another context kept the GPU busy -- which is exactly the case
// of one thread encoding and another decoding (both PCIe directions in use).
// With pageable host memory the copies degrade to synchronous ones but stay correct.
template <class FIn, class FRun, class FOut>
int run_pipeline_steps(himgcu_ctx *ctx, int K, int S, cudaStream_t q_in, cudaStream_t q_out, FIn copy_in, FRun run, FOut copy_out) {
  int n_in = 0, n_run = 0, n_out = 0;  // sub-batches copied in / launched / drained so far
  auto done = [&](cudaEvent_t e, bool *ok) -> int {
    const cudaError_t q = cudaEventQuery(e);
    if (q != cudaSuccess && q != cudaErrorNotReady) CK(q);
    *ok = q == cudaSuccess;
    return HIMGCU_OK;
  };
  while (n_out < K) {
    bool progressed = false, ok = false;
    int rc;
    if (n_out < n_run) {  // coded -> copy out
      const int b = n_out % S;
      if ((rc = done(ctx->ev_cmp[b], &ok))) return rc;
      if (ok) {
        if ((rc = copy_out(n_out, b))) return rc;
        CK(cudaEventRecord(ctx->ev_out[b], q_out));
        ++n_out;
        progressed = true;
      }
    }
    if (n_run < n_in) {  // copied in (and the slot's previous output drained) -> launch
      const int b = n_run % S;
      if ((rc = done(ctx->ev_in[b], &ok))) return rc;
      if (ok && n_run >= S && (rc = done(ctx->ev_out[b], &ok))) return rc;
      if (ok) {
        himgcu_ctx *L = lane_of(ctx, b);
        if ((rc = run(n_run, b, L))) {
          if (L != ctx) ctx->err = L->err;
          return rc;
        }
        CK(cudaEventRecord(ctx->ev_cmp[b], L->stream));
        ++n_run;
        progressed = true;
      }
    }
    if (n_in < K && n_in < n_out + S && n_in < n_run + 2) {  // slot free -> copy in (at most 2 ahead)
      const int b = n_in % S;
      if ((rc = copy_in(n_in, b))) return rc;
      CK(cudaEventRecord(ctx->ev_in[b], q_in));
      ++n_in;
      progressed = true;
    }
    if (!progressed) std::this_thread::sleep_for(std::chrono::microseconds(20));
  }
  if (K > 0) CK(cudaEventSynchronize(ctx->ev_out[(K - 1) % S]));  // own copies only: the queue is shared
  return finish_lanes(ctx, S);
}

// An error leaves sub-batches in flight (lanes still coding, copies queued on the shared streams that
// write into the caller's buffers): drain everything before the caller sees the error and may free or
// reuse its buffers.
template <class FIn, class FRun, class FOut>
int run_pipeline(himgcu_ctx *ctx, int K, int S, cudaStream_t q_in, cudaStream_t q_out, FIn copy_in, FRun run, FOut copy_out) {
  const int rc = run_pipeline_steps(ctx, K, S, q_in, q_out, copy_in, run, copy_out);
  if (rc != HIMGCU_OK) {
    const std::string why = ctx->err;
    for (int b = 0; b < S; ++b) cudaStreamSynchronize(lane_of(ctx, b)->stream);
    cudaStreamSynchronize(q_in);
    cudaStreamSynchronize(q_out);
    finish_lanes(ctx, S);
    cudaGetLastError();
    ctx->err = why;
  }
  return rc;
}

}  // namespace

// ================================================================================================
extern "C" {

int himgcu_abi_version(void) { return 1; }

int himgcu_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

int himgcu_create(int device, himgcu_ctx **out) {
  if (!out) return HIMGCU_ERR_ARG;
  *out = nullptr;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || device < 0 || device >= n) return HIMGCU_ERR_CUDA;
  if (cudaSetDevice(device) != cudaSuccess) return HIMGCU_ERR_CUDA;
  himgcu_ctx *ctx = new himgcu_ctx();
  ctx->device = device;
  if (cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking) != cudaSuccess) {
    delete ctx;
    return HIMGCU_ERR_CUDA;
  }
  ctx->stream = ctx->own_stream;
  if (const char *v = getenv("HIMG_XFORM_VARIANT")) ctx->xform_variant = atoi(v);  // experiments only
  *out = ctx;
  return HIMGCU_OK;
}

void himgcu_destroy(himgcu_ctx *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  resolve_profile(ctx);
  for (auto &kv : ctx->bufs)
    if (kv.second.p) cudaFree(kv.second.p);
  if (ctx->full_lut.p) cudaFree(ctx->full_lut.p);
  if (ctx->signed_lut.p) cudaFree(ctx->signed_lut.p);
  if (ctx->pinned) cudaFreeHost(ctx->pinned);
  for (int k = 0; k < 2; ++k) {
    if (ctx->stage[k]) cudaFreeHost(ctx->stage[k]);
    if (ctx->stage_ev[k]) cudaEventDestroy(ctx->stage_ev[k]);
  }
  for (cudaEvent_t e : ctx->event_pool) cudaEventDestroy(e);
  for (himgcu_ctx *l : ctx->lanes) himgcu_destroy(l);
  for (int b = 0; b < himgcu_ctx::kMaxLanes; ++b) {
    if (ctx->ev_in[b]) cudaEventDestroy(ctx->ev_in[b]);
    if (ctx->ev_cmp[b]) cudaEventDestroy(ctx->ev_cmp[b]);
    if (ctx->ev_out[b]) cudaEventDestroy(ctx->ev_out[b]);
  }
  // in_stream / out_stream are the process-wide copy queues: not destroyed here
  if (ctx->aux_stream) cudaStreamDestroy(ctx->aux_stream);
  if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
  if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
  if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
  delete ctx;
}

int himgcu_set_stream(himgcu_ctx *ctx, void *cuda_stream) {
  if (!ctx) return HIMGCU_ERR_ARG;
  if (ctx->stream == reinterpret_cast<cudaStream_t>(cuda_stream)) return HIMGCU_OK;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);  // the context's scratch buffers are reused by the next call
  ctx->stream = reinterpret_cast<cudaStream_t>(cuda_stream);
  return HIMGCU_OK;
}

int himgcu_reset_stream(himgcu_ctx *ctx) {
  if (!ctx) return HIMGCU_ERR_ARG;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  ctx->stream = ctx->own_stream;
  return HIMGCU_OK;
}

int himgcu_synchronize(himgcu_ctx *ctx) {
  if (!ctx) return HIMGCU_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  CK(cudaStreamSynchronize(ctx->stream));
  resolve_profile(ctx);
  return HIMGCU_OK;
}

const char *himgcu_last_error(himgcu_ctx *ctx) { return ctx ? ctx->err.c_str() : "null context"; }

uint64_t himgcu_fnv1a64(const uint8_t *data, size_t size) {
  // offset basis exactly as in SURVEY.md Appendix B (the recorded reference hashes were made with it)
  uint64_t h = 1469598103934665603ull;
  for (size_t i = 0; i < size; ++i) h = (h ^ data[i]) * 1099511628211ull;
  return h;
}

size_t himgcu_encode_bound(int w, int h, int nch) {
  if (!shape_ok(w, h, nch)) return 0;
  const Geom g = make_geom(w, h, nch, nch);
  // RIFF(12) FRMT(19) LMAP(136) LRES hdr(8) QCFG(72) FMAP(188) FRES hdr(8) + two Huffman chunks.  A
  // Huffman code over the 261 symbols spends less than log2(261) + 1 < 9.03 bits per token and a token
  // covers at least one byte, so a chunk of n bytes packs into less than n + n/7 bytes, plus its tree
  // (<= 359 bytes), one byte of padding and a 2/4-byte header per segment.  (The reference sizes its
  // buffer as n + 359, huffman_enc.cpp:242-244, which incompressible data can overflow.)
  const size_t lres = (size_t)g.lres_size, fres = (size_t)g.planes_bytes;
  return 12 + 19 + 136 + 8 + 72 + 188 + 8 + (lres + lres / 7 + 359 + 8) + (fres + fres / 7 + 359 + (size_t)5 * g.rows) + 64;
}

size_t himgcu_lres_size(int w, int h, int nch) { return shape_ok(w, h, nch) ? (size_t)make_geom(w, h, nch, nch).lres_size : 0; }
size_t himgcu_lres_stride(int w, int h, int nch) { return shape_ok(w, h, nch) ? (size_t)make_geom(w, h, nch, nch).lres_stride : 0; }

int himgcu_encode_batch(himgcu_ctx *ctx, const uint8_t *d_pixels, int n, int w, int h, int nch, int quality,
                        int use_ycbcr, uint8_t *d_out, size_t out_stride, uint32_t *d_sizes) {
  if (!ctx || !d_pixels || !d_out || !d_sizes || n < 0) return fail(ctx, HIMGCU_ERR_ARG, "bad argument");
  if (!shape_ok(w, h, nch)) return fail(ctx, HIMGCU_ERR_UNSUPPORTED, "unsupported shape %dx%dx%d", w, h, nch);
  if (n == 0) return HIMGCU_OK;
  CK(cudaSetDevice(ctx->device));
  const Geom g = make_geom(w, h, nch, nch);
  const bool ycbcr = use_ycbcr && nch >= 3;
  return for_sub_batches(ctx, n, per_image_encode_ws(g), [&](int i0, int m) -> int {
    return encode_device(ctx, d_pixels + (size_t)i0 * g.img_bytes, m, g, quality, ycbcr, d_out + (size_t)i0 * out_stride,
                         out_stride, d_sizes + i0);
  });
}

int himgcu_encode_batch_mixed(himgcu_ctx *ctx, const uint8_t *d_pixels, const uint64_t *d_pixel_offsets, const int32_t *d_dims,
                              int n, int max_width, int max_height, int nch, int quality, int use_ycbcr, uint8_t *d_out,
                              size_t out_stride, uint32_t *d_sizes) {
  if (!ctx || !d_pixels || !d_pixel_offsets || !d_dims || !d_out || !d_sizes || n < 0) return fail(ctx, HIMGCU_ERR_ARG, "bad argument");
  if (!shape_ok(max_width, max_height, nch))
    return fail(ctx, HIMGCU_ERR_UNSUPPORTED, "unsupported bounding shape %dx%dx%d", max_width, max_height, nch);
  if (n == 0) return HIMGCU_OK;
  CK(cudaSetDevice(ctx->device));
  // every per-image scratch slot has the bounding geometry's size; the kernels lay each image out in its own
  const Geom g = make_geom(max_width, max_height, nch, nch);
  const bool ycbcr = use_ycbcr && nch >= 3;
  return for_sub_batches(ctx, n, per_image_encode_ws(g), [&](int i0, int m) -> int {
    const MixedDims md{d_dims + 2 * (size_t)i0, max_width, max_height, nch};
    return encode_device<true>(ctx, d_pixels, m, g, quality, ycbcr, d_out + (size_t)i0 * out_stride, out_stride, d_sizes + i0, md,
                               reinterpret_cast<const unsigned long long *>(d_pixel_offsets) + i0);
  });
}

}  // extern "C"

namespace {

// Is `p` page-locked host memory (cudaMallocHost / cudaHostRegister / himgcu_host_alloc)?
bool is_pinned(const void *p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeHost;
}

// Single-image host calls move up to tens of megabytes through PCIe.  Page-locked caller memory is
// copied directly (asynchronously, at link speed).  Pageable memory goes through two page-locked
// staging slots owned by the context, so that the CPU copy of chunk k overlaps the DMA of chunk k-1
// (a plain cudaMemcpyAsync from pageable memory is staged by the driver in one blocking piece).
constexpr size_t kStageChunk = (size_t)4 << 20;

int ensure_stage(himgcu_ctx *ctx) {
  if (!ctx->stage[0]) {
    for (int k = 0; k < 2; ++k) {
      CK(cudaMallocHost(&ctx->stage[k], kStageChunk));
      CK(cudaEventCreateWithFlags(&ctx->stage_ev[k], cudaEventDisableTiming));
    }
  }
  return HIMGCU_OK;
}

int copy_to_device(himgcu_ctx *ctx, void *dst, const void *src, size_t bytes) {
  if (bytes <= (64 << 10) || is_pinned(src)) {
    CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return HIMGCU_OK;
  }
  int rc = ensure_stage(ctx);
  if (rc) return rc;
  int k = 0;
  for (size_t off = 0; off < bytes; off += kStageChunk, k ^= 1) {
    const size_t m = std::min(kStageChunk, bytes - off);
    CK(cudaEventSynchronize(ctx->stage_ev[k]));  // the slot's previous DMA is done
    memcpy(ctx->stage[k], (const char *)src + off, m);
    CK(cudaMemcpyAsync((char *)dst + off, ctx->stage[k], m, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaEventRecord(ctx->stage_ev[k], ctx->stream));
  }
  return HIMGCU_OK;
}

// Device -> host; returns after the data has arrived.
int copy_to_host(himgcu_ctx *ctx, void *dst, const void *src, size_t bytes) {
  if (bytes <= (64 << 10) || is_pinned(dst)) {
    CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return HIMGCU_OK;
  }
  int rc = ensure_stage(ctx);
  if (rc) return rc;
  size_t off_prev = 0, m_prev = 0;
  int k = 0;
  for (size_t off = 0; off < bytes; off += kStageChunk, k ^= 1) {
    const size_t m = std::min(kStageChunk, bytes - off);
    CK(cudaMemcpyAsync(ctx->stage[k], (const char *)src + off, m, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaEventRecord(ctx->stage_ev[k], ctx->stream));
    if (m_prev) {  // drain the other slot while this chunk is on the wire
      CK(cudaEventSynchronize(ctx->stage_ev[k ^ 1]));
      memcpy((char *)dst + off_prev, ctx->stage[k ^ 1], m_prev);
    }
    off_prev = off;
    m_prev = m;
  }
  if (m_prev) {
    CK(cudaEventSynchronize(ctx->stage_ev[k ^ 1]));
    memcpy((char *)dst + off_prev, ctx->stage[k ^ 1], m_prev);
  }
  return HIMGCU_OK;
}

// log2 of the factor of a scaled decode: 0 to 3 for 1, 2, 4, 8; -1 for any other factor.
int scale_log2(int factor) {
  switch (factor) {
    case 1: return 0;
    case 2: return 1;
    case 4: return 2;
    case 8: return 3;
    default: return -1;
  }
}

// Bytes of one image of g decoded at 1 / 2^lf size: [ceil(h / 2^lf)][ceil(w / 2^lf)][nch].
size_t scaled_bytes(const Geom &g, int lf) {
  const int f = 1 << lf;
  return (size_t)((g.w + f - 1) >> lf) * (size_t)((g.h + f - 1) >> lf) * (size_t)g.nch;
}

// himgcu_decode_batch(_scaled), and with MIXED himgcu_decode_batch_mixed(_scaled), whose w x h are the bounds of the
// images: image i goes to d_pixels_out + i * scaled_bytes(g, lf), or with MIXED to d_pixels_out + d_pixel_offsets[i].
template <bool MIXED>
int decode_batch_lf(himgcu_ctx *ctx, const uint8_t *d_himg, const uint64_t *d_offsets, const uint32_t *d_sizes, int n,
                    const int32_t *d_dims, int w, int h, int nch, int flags, int lf, const uint64_t *d_pixel_offsets,
                    uint8_t *d_pixels_out, int32_t *d_status) {
  if (!ctx || !d_himg || !d_offsets || !d_sizes || (MIXED && (!d_dims || !d_pixel_offsets)) || !d_pixels_out || !d_status || n < 0)
    return fail(ctx, HIMGCU_ERR_ARG, "bad argument");
  if (!shape_ok(w, h, nch))
    return fail(ctx, HIMGCU_ERR_UNSUPPORTED, "unsupported %sshape %dx%dx%d", MIXED ? "bounding " : "", w, h, nch);
  if (n == 0) return HIMGCU_OK;
  CK(cudaSetDevice(ctx->device));
  // with MIXED every per-image scratch slot has the bounding geometry's size; the kernels lay each image out in its own
  const Geom g = make_geom(w, h, nch, nch);
  const size_t per = per_image_encode_ws(g) + sizeof(DecTables) + 2 * sizeof(DecTree);
  return for_sub_batches(ctx, n, per, [&](int i0, int m) -> int {
    const MixedDims md = MIXED ? MixedDims{d_dims + 2 * (size_t)i0, w, h, nch} : MixedDims{};
    const unsigned long long *px_off = MIXED ? reinterpret_cast<const unsigned long long *>(d_pixel_offsets) + i0 : nullptr;
    uint8_t *out = MIXED ? d_pixels_out : d_pixels_out + (size_t)i0 * scaled_bytes(g, lf);
    return decode_device<MIXED>(ctx, d_himg, reinterpret_cast<const unsigned long long *>(d_offsets) + i0, d_sizes + i0, m, g, flags,
                                out, d_status + i0, lf, md, px_off);
  });
}

// himgcu_decode_batch_region(_scaled), and with MIXED himgcu_decode_batch_region_mixed(_scaled), whose w x h are the
// bounds of the images.  lf > 0: the rectangles are those of the images scaled by 2^lf, and rw x rh must fit the
// scaled bounds.
template <bool MIXED>
int decode_batch_region(himgcu_ctx *ctx, const uint8_t *d_himg, const uint64_t *d_offsets, const uint32_t *d_sizes, int n,
                        const int32_t *d_dims, int w, int h, int nch, int flags, int lf, const int32_t *d_origins, int rw, int rh,
                        uint8_t *d_pixels_out, int32_t *d_status) {
  if (!ctx || !d_himg || !d_offsets || !d_sizes || (MIXED && !d_dims) || !d_origins || !d_pixels_out || !d_status || n < 0)
    return fail(ctx, HIMGCU_ERR_ARG, "bad argument");
  if (!shape_ok(w, h, nch))
    return fail(ctx, HIMGCU_ERR_UNSUPPORTED, "unsupported %sshape %dx%dx%d", MIXED ? "bounding " : "", w, h, nch);
  const int sw = (w + (1 << lf) - 1) >> lf, sh = (h + (1 << lf) - 1) >> lf;  // the (scaled) bounds of a rectangle
  if (rw < 1 || rh < 1 || rw > sw || rh > sh)
    return fail(ctx, HIMGCU_ERR_ARG, MIXED ? "region %dx%d does not fit the %dx%d bounds" : "region %dx%d does not fit a %dx%d image",
                rw, rh, sw, sh);
  if (n == 0) return HIMGCU_OK;
  CK(cudaSetDevice(ctx->device));
  const Geom g = make_geom(w, h, nch, nch);
  const int kr = region_rows(g, rh, lf);
  const size_t out_bytes = (size_t)rw * rh * nch;
  // (the uniform count includes the tables of the lane-pair inverse, which a mixed batch does not take)
  const size_t per = per_image_encode_ws(g) - g.planes_bytes + (size_t)kr * (g.seg + sizeof(SegRef)) + sizeof(DecTables) +
                     2 * sizeof(DecTree) + (MIXED ? 0 : sizeof(InvTables));
  return for_sub_batches(ctx, n, per, [&](int i0, int m) -> int {
    const MixedDims md = MIXED ? MixedDims{d_dims + 2 * (size_t)i0, w, h, nch} : MixedDims{};
    return decode_region_device<MIXED>(ctx, d_himg, reinterpret_cast<const unsigned long long *>(d_offsets) + i0, d_sizes + i0, m,
                                       g, flags, d_origins + 2 * (size_t)i0, rw, rh, d_pixels_out + (size_t)i0 * out_bytes,
                                       d_status + i0, md, lf);
  });
}

struct Rect {
  int x, y, w, h;
};

// himgcu_decode, himgcu_decode_scaled (lf > 0, out_cap is checked against the scaled size) and, with `rect`,
// himgcu_decode_region(_scaled) (a rectangle of the image scaled by 2^lf).
int decode_single(himgcu_ctx *ctx, const uint8_t *himg, size_t size, int flags, int lf, const Rect *rect, uint8_t *out,
                  size_t out_cap, int *w, int *h, int *nch) {
  if (!ctx || !himg || !out) return fail(ctx, HIMGCU_ERR_ARG, "bad argument");
  int W = 0, H = 0, N = 0;
  if (himgcu_decode_info(himg, size, &W, &H, &N) != HIMGCU_OK) return fail(ctx, HIMGCU_REJECT, "not a HIMG stream");
  if (w) *w = W;
  if (h) *h = H;
  if (nch) *nch = N;
  if (W < 1 || H < 1 || N < 1) return fail(ctx, HIMGCU_REJECT, "bad dimensions");
  if (!shape_ok(W, H, N)) return fail(ctx, HIMGCU_ERR_UNSUPPORTED, "unsupported shape %dx%dx%d", W, H, N);
  if (size > 0xffffffffull) return fail(ctx, HIMGCU_ERR_UNSUPPORTED, "stream too large");
  const int SW = (W + (1 << lf) - 1) >> lf, SH = (H + (1 << lf) - 1) >> lf;  // the scaled image
  if (rect && (rect->w < 1 || rect->h < 1 || rect->x < 0 || rect->y < 0 || rect->x > SW - rect->w || rect->y > SH - rect->h))
    return fail(ctx, HIMGCU_ERR_ARG, "region %dx%d at (%d, %d) is empty or outside the %dx%d image", rect->w, rect->h, rect->x,
                rect->y, SW, SH);
  CK(cudaSetDevice(ctx->device));
  const Geom g = make_geom(W, H, N, N);
  const size_t out_bytes = rect ? (size_t)rect->w * rect->h * N : scaled_bytes(g, lf);
  if (out_bytes > out_cap) return fail(ctx, HIMGCU_ERR_CAPACITY, "output buffer too small");
  uint8_t *d_in, *d_px;
  unsigned long long *d_off;
  uint32_t *d_sz;
  int *d_status;
  int32_t *d_org = nullptr;
  ENSURE("single_in", size + 16, d_in);
  ENSURE(rect ? "single_rpx" : "single_px", out_bytes, d_px);
  ENSURE("single_off", sizeof(unsigned long long), d_off);
  ENSURE("single_size", sizeof(uint32_t), d_sz);
  ENSURE("single_status", sizeof(int), d_status);
  if (rect) ENSURE("single_origin", 2 * sizeof(int32_t), d_org);
  int rc = ensure_pinned(ctx, 64);
  if (rc) return rc;
  // offset / size / status / origin travel through the context's page-locked scratch (truly asynchronous copies)
  unsigned long long *h_off = reinterpret_cast<unsigned long long *>(ctx->pinned);
  uint32_t *h_sz = reinterpret_cast<uint32_t *>(h_off + 1);
  int *h_status = reinterpret_cast<int *>(h_off + 2);
  int32_t *h_org = reinterpret_cast<int32_t *>(h_off + 3);
  CK(cudaStreamSynchronize(ctx->stream));  // (the scratch words of the previous call are no longer in flight)
  *h_off = 0;
  *h_sz = (uint32_t)size;
  if (rect) {
    h_org[0] = rect->x;
    h_org[1] = rect->y;
  }
  if ((rc = copy_to_device(ctx, d_in, himg, size))) return rc;
  CK(cudaMemcpyAsync(d_off, h_off, sizeof(*h_off), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(d_sz, h_sz, sizeof(*h_sz), cudaMemcpyHostToDevice, ctx->stream));
  if (rect) {
    CK(cudaMemcpyAsync(d_org, h_org, 2 * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
    rc = decode_region_device(ctx, d_in, d_off, d_sz, 1, g, flags, d_org, rect->w, rect->h, d_px, d_status, {}, lf);
  } else {
    rc = decode_device(ctx, d_in, d_off, d_sz, 1, g, flags, d_px, d_status, lf);
  }
  if (rc) return rc;
  // The pixels follow the status on the same stream without a round trip in between: a rejected stream
  // costs one wasted copy, an accepted one (the common case) saves a synchronisation.
  CK(cudaMemcpyAsync(h_status, d_status, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  if ((rc = copy_to_host(ctx, out, d_px, out_bytes))) return rc;
  if (*h_status) return fail(ctx, HIMGCU_REJECT, "stream rejected");
  return HIMGCU_OK;
}

}  // namespace

extern "C" {

int himgcu_encode(himgcu_ctx *ctx, const uint8_t *pixels, int w, int h, int pixel_stride, int nch, int quality,
                  int use_ycbcr, uint8_t *out, size_t out_cap, size_t *out_size) {
  if (!ctx || !pixels || !out || !out_size) return fail(ctx, HIMGCU_ERR_ARG, "bad argument");
  if (!shape_ok(w, h, nch) || pixel_stride < nch || pixel_stride > 64)
    return fail(ctx, HIMGCU_ERR_UNSUPPORTED, "unsupported shape %dx%dx%d stride %d", w, h, nch, pixel_stride);
  CK(cudaSetDevice(ctx->device));
  *out_size = 0;
  const Geom g = make_geom(w, h, nch, pixel_stride);
  const bool ycbcr = use_ycbcr && nch >= 3;
  const size_t bound = himgcu_encode_bound(w, h, nch);
  uint8_t *d_in, *d_out;
  uint32_t *d_size;
  ENSURE("single_in", g.img_bytes, d_in);
  ENSURE("single_out", bound, d_out);
  ENSURE("single_size", sizeof(uint32_t), d_size);
  int rc = copy_to_device(ctx, d_in, pixels, g.img_bytes);
  if (rc) return rc;
  rc = encode_device(ctx, d_in, 1, g, quality, ycbcr, d_out, bound, d_size);
  if (rc) return rc;
  // one round trip for the size and the encoder's status flag (read = clear)
  rc = ensure_pinned(ctx, 64);
  if (rc) return rc;
  uint32_t *h_size = reinterpret_cast<uint32_t *>(ctx->pinned);
  int *h_err = reinterpret_cast<int *>(ctx->pinned) + 1, *d_err;
  ENSURE("enc_err", sizeof(int), d_err);
  CK(cudaMemcpyAsync(h_size, d_size, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(h_err, d_err, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemsetAsync(d_err, 0, sizeof(int), ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  const uint32_t size = *h_size;
  if ((rc = enc_err_status(ctx, *h_err))) return rc;
  if (size == 0) return fail(ctx, HIMGCU_ERR_CAPACITY, "internal output bound exceeded");
  if (size > out_cap) return fail(ctx, HIMGCU_ERR_CAPACITY, "output buffer too small: need %u", size);
  if ((rc = copy_to_host(ctx, out, d_out, size))) return rc;
  *out_size = size;
  return HIMGCU_OK;
}

int himgcu_decode_info(const uint8_t *p, size_t size, int *w, int *h, int *nch) {
  if (!p || size < 12 || memcmp(p, "RIFF", 4) || memcmp(p + 8, "HIMG", 4)) return HIMGCU_REJECT;
  auto u32 = [&](size_t o) { return (uint32_t)p[o] | ((uint32_t)p[o + 1] << 8) | ((uint32_t)p[o + 2] << 16) | ((uint32_t)p[o + 3] << 24); };
  if ((long long)(int)u32(4) + 8 != (long long)size) return HIMGCU_REJECT;
  size_t idx = 12;
  for (;;) {
    if (idx + 8 > size) return HIMGCU_REJECT;
    const uint32_t cc = u32(idx);
    const int sz = (int)u32(idx + 4);
    idx += 8;
    if (sz < 0 || idx + (size_t)sz > size) return HIMGCU_REJECT;
    if (cc == 0x544d5246u) {
      if (sz < 11 || p[idx] != 1) return HIMGCU_REJECT;
      if (w) *w = (int)u32(idx + 1);
      if (h) *h = (int)u32(idx + 5);
      if (nch) *nch = p[idx + 9];
      return HIMGCU_OK;
    }
    idx += sz;
  }
}

int himgcu_decode_batch(himgcu_ctx *ctx, const uint8_t *d_himg, const uint64_t *d_offsets, const uint32_t *d_sizes,
                        int n, int w, int h, int nch, int flags, uint8_t *d_pixels_out, int32_t *d_status) {
  return decode_batch_lf<false>(ctx, d_himg, d_offsets, d_sizes, n, nullptr, w, h, nch, flags, 0, nullptr, d_pixels_out, d_status);
}

int himgcu_decode_batch_scaled(himgcu_ctx *ctx, const uint8_t *d_himg, const uint64_t *d_offsets, const uint32_t *d_sizes,
                               int n, int w, int h, int nch, int flags, int factor, uint8_t *d_pixels_out, int32_t *d_status) {
  const int lf = scale_log2(factor);
  if (lf < 0) return fail(ctx, HIMGCU_ERR_ARG, "scale factor %d is not 1, 2, 4 or 8", factor);
  return decode_batch_lf<false>(ctx, d_himg, d_offsets, d_sizes, n, nullptr, w, h, nch, flags, lf, nullptr, d_pixels_out, d_status);
}

int himgcu_decode_batch_mixed(himgcu_ctx *ctx, const uint8_t *d_himg, const uint64_t *d_offsets, const uint32_t *d_sizes, int n,
                              const int32_t *d_dims, int max_width, int max_height, int nch, int flags,
                              const uint64_t *d_pixel_offsets, uint8_t *d_pixels_out, int32_t *d_status) {
  return decode_batch_lf<true>(ctx, d_himg, d_offsets, d_sizes, n, d_dims, max_width, max_height, nch, flags, 0, d_pixel_offsets,
                               d_pixels_out, d_status);
}

int himgcu_decode_batch_mixed_scaled(himgcu_ctx *ctx, const uint8_t *d_himg, const uint64_t *d_offsets, const uint32_t *d_sizes,
                                     int n, const int32_t *d_dims, int max_width, int max_height, int nch, int flags, int factor,
                                     const uint64_t *d_pixel_offsets, uint8_t *d_pixels_out, int32_t *d_status) {
  const int lf = scale_log2(factor);
  if (lf < 0) return fail(ctx, HIMGCU_ERR_ARG, "scale factor %d is not 1, 2, 4 or 8", factor);
  return decode_batch_lf<true>(ctx, d_himg, d_offsets, d_sizes, n, d_dims, max_width, max_height, nch, flags, lf, d_pixel_offsets,
                               d_pixels_out, d_status);
}

int himgcu_decode(himgcu_ctx *ctx, const uint8_t *himg, size_t size, int flags, uint8_t *out, size_t out_cap, int *w,
                  int *h, int *nch) {
  return decode_single(ctx, himg, size, flags, 0, nullptr, out, out_cap, w, h, nch);
}

int himgcu_decode_scaled(himgcu_ctx *ctx, const uint8_t *himg, size_t size, int flags, int factor, uint8_t *out, size_t out_cap,
                         int *w, int *h, int *nch) {
  const int lf = scale_log2(factor);
  if (lf < 0) return fail(ctx, HIMGCU_ERR_ARG, "scale factor %d is not 1, 2, 4 or 8", factor);
  return decode_single(ctx, himg, size, flags, lf, nullptr, out, out_cap, w, h, nch);
}

int himgcu_decode_batch_region(himgcu_ctx *ctx, const uint8_t *d_himg, const uint64_t *d_offsets, const uint32_t *d_sizes, int n,
                               int w, int h, int nch, int flags, const int32_t *d_origins, int rw, int rh, uint8_t *d_pixels_out,
                               int32_t *d_status) {
  return decode_batch_region<false>(ctx, d_himg, d_offsets, d_sizes, n, nullptr, w, h, nch, flags, 0, d_origins, rw, rh,
                                    d_pixels_out, d_status);
}

int himgcu_decode_batch_region_scaled(himgcu_ctx *ctx, const uint8_t *d_himg, const uint64_t *d_offsets, const uint32_t *d_sizes,
                                      int n, int w, int h, int nch, int flags, int factor, const int32_t *d_origins, int rw, int rh,
                                      uint8_t *d_pixels_out, int32_t *d_status) {
  const int lf = scale_log2(factor);
  if (lf < 0) return fail(ctx, HIMGCU_ERR_ARG, "scale factor %d is not 1, 2, 4 or 8", factor);
  return decode_batch_region<false>(ctx, d_himg, d_offsets, d_sizes, n, nullptr, w, h, nch, flags, lf, d_origins, rw, rh,
                                    d_pixels_out, d_status);
}

int himgcu_decode_batch_region_mixed(himgcu_ctx *ctx, const uint8_t *d_himg, const uint64_t *d_offsets, const uint32_t *d_sizes,
                                     int n, const int32_t *d_dims, int max_width, int max_height, int nch, int flags,
                                     const int32_t *d_origins, int rw, int rh, uint8_t *d_pixels_out, int32_t *d_status) {
  return decode_batch_region<true>(ctx, d_himg, d_offsets, d_sizes, n, d_dims, max_width, max_height, nch, flags, 0, d_origins, rw,
                                   rh, d_pixels_out, d_status);
}

int himgcu_decode_batch_region_mixed_scaled(himgcu_ctx *ctx, const uint8_t *d_himg, const uint64_t *d_offsets,
                                            const uint32_t *d_sizes, int n, const int32_t *d_dims, int max_width, int max_height,
                                            int nch, int flags, int factor, const int32_t *d_origins, int rw, int rh,
                                            uint8_t *d_pixels_out, int32_t *d_status) {
  const int lf = scale_log2(factor);
  if (lf < 0) return fail(ctx, HIMGCU_ERR_ARG, "scale factor %d is not 1, 2, 4 or 8", factor);
  return decode_batch_region<true>(ctx, d_himg, d_offsets, d_sizes, n, d_dims, max_width, max_height, nch, flags, lf, d_origins, rw,
                                   rh, d_pixels_out, d_status);
}

int himgcu_decode_region(himgcu_ctx *ctx, const uint8_t *himg, size_t size, int flags, int x, int y, int rw, int rh, uint8_t *out,
                         size_t out_cap, int *w, int *h, int *nch) {
  const Rect rect{x, y, rw, rh};
  return decode_single(ctx, himg, size, flags, 0, &rect, out, out_cap, w, h, nch);
}

int himgcu_decode_region_scaled(himgcu_ctx *ctx, const uint8_t *himg, size_t size, int flags, int factor, int x, int y, int rw,
                                int rh, uint8_t *out, size_t out_cap, int *w, int *h, int *nch) {
  const int lf = scale_log2(factor);
  if (lf < 0) return fail(ctx, HIMGCU_ERR_ARG, "scale factor %d is not 1, 2, 4 or 8", factor);
  const Rect rect{x, y, rw, rh};
  return decode_single(ctx, himg, size, flags, lf, &rect, out, out_cap, w, h, nch);
}

// ---- batch with host buffers -------------------------------------------------------------------

void *himgcu_host_alloc(size_t bytes) {
  void *p = nullptr;
  if (cudaMallocHost(&p, bytes) != cudaSuccess) return nullptr;
  return p;
}

void himgcu_host_free(void *p) {
  if (p) cudaFreeHost(p);
}

int himgcu_encode_batch_host(himgcu_ctx *ctx, const uint8_t *pixels, int n, int w, int h, int nch, int quality,
                             int use_ycbcr, uint8_t *out, size_t out_cap, uint64_t *offsets, uint32_t *sizes) {
  if (!ctx || !pixels || !out || !offsets || !sizes || n < 0) return fail(ctx, HIMGCU_ERR_ARG, "bad argument");
  if (!shape_ok(w, h, nch)) return fail(ctx, HIMGCU_ERR_UNSUPPORTED, "unsupported shape %dx%dx%d", w, h, nch);
  CK(cudaSetDevice(ctx->device));
  int rc = ensure_pipeline(ctx);
  if (rc) return rc;
  const Geom g = make_geom(w, h, nch, nch);
  const bool ycbcr = use_ycbcr && nch >= 3;
  const size_t stride = (himgcu_encode_bound(w, h, nch) + 255) & ~(size_t)255;
  int sub = (int)std::max<size_t>(1, std::min<size_t>((size_t)std::max(n, 1), ctx->host_sub_bytes / (g.img_bytes + stride)));
  sub = std::min(sub, 65535);
  const int K = (n + sub - 1) / sub;
  int S = 1;
  if ((rc = prepare_lanes(ctx, K, &S))) return rc;
  uint8_t *d_in[himgcu_ctx::kMaxLanes], *d_out[himgcu_ctx::kMaxLanes];
  uint32_t *d_sizes[himgcu_ctx::kMaxLanes], *h_sizes[himgcu_ctx::kMaxLanes];
  for (int b = 0; b < S; ++b) {
    const std::string sfx = std::to_string(b);
    ENSURE(("hb_in" + sfx).c_str(), (size_t)sub * g.img_bytes, d_in[b]);
    ENSURE(("hb_out" + sfx).c_str(), (size_t)sub * stride, d_out[b]);
    ENSURE(("hb_sizes" + sfx).c_str(), (size_t)sub * sizeof(uint32_t), d_sizes[b]);
  }
  rc = ensure_pinned(ctx, (size_t)S * sub * sizeof(uint32_t));
  if (rc) return rc;
  for (int b = 0; b < S; ++b) h_sizes[b] = reinterpret_cast<uint32_t *>(ctx->pinned) + (size_t)b * sub;
  cudaStream_t s_in = ctx->in_stream, s_out = ctx->out_stream;
  for (int b = 0; b < S; ++b) CK(cudaStreamSynchronize(lane_of(ctx, b)->stream));
  PipeTrace trace("enc");
  uint64_t pos = 0;
  offsets[0] = 0;
  int failed_image = -1;
  rc = run_pipeline(
      ctx, K, S, s_in, s_out,
      [&](int k, int b) -> int {
        const int i0 = k * sub, m = std::min(sub, n - i0);
        trace.mark(k, 0, s_in);
        CK(cudaMemcpyAsync(d_in[b], pixels + (size_t)i0 * g.img_bytes, (size_t)m * g.img_bytes, cudaMemcpyHostToDevice, s_in));
        trace.mark(k, 1, s_in);
        return HIMGCU_OK;
      },
      [&](int k, int b, himgcu_ctx *L) -> int {
        const int m = std::min(sub, n - k * sub);
        trace.launched(k);
        int r = encode_device(L, d_in[b], m, g, quality, ycbcr, d_out[b], stride, d_sizes[b]);
        if (r) return r;
        // The sizes reach the host by a KERNEL that stores them into the page-locked array, not by a copy on
        // the lane's stream: a device-to-host copy from this stream was measured to wait for tens of
        // milliseconds while another context (a decode call in another thread) kept the copy engine of
        // that direction busy from its own stream.
        k_store_u32<<<(m + 255) / 256, 256, 0, L->stream>>>(h_sizes[b], d_sizes[b], m);
        if (cudaGetLastError() != cudaSuccess) return fail(L, HIMGCU_ERR_CUDA, "size read-back failed");
        trace.mark(k, 2, L->stream);
        return HIMGCU_OK;
      },
      [&](int k, int b) -> int {
        const int i0 = k * sub, m = std::min(sub, n - i0);
        for (int i = 0; i < m; ++i) {  // the sizes of sub-batch k are on the host
          const uint32_t sz = h_sizes[b][i];
          sizes[i0 + i] = sz;
          if (sz == 0) {
            failed_image = i0 + i;
            return fail(ctx, HIMGCU_ERR_CAPACITY, "image %d could not be encoded", i0 + i);
          }
          if (pos + sz > out_cap) return fail(ctx, HIMGCU_ERR_CAPACITY, "output buffer too small");
          CK(cudaMemcpyAsync(out + pos, d_out[b] + (size_t)i * stride, sz, cudaMemcpyDeviceToHost, s_out));
          pos += ((uint64_t)sz + 15) & ~15ull;
          offsets[i0 + i + 1] = pos;
        }
        trace.mark(k, 3, s_out);
        return HIMGCU_OK;
      });
  // the device flags of the lanes say why an image was not encoded (and catch an internal mismatch even
  // when every size is non-zero)
  for (int b = 0; b < S; ++b) {
    himgcu_ctx *L = lane_of(ctx, b);
    if (L->bufs.find("enc_err") == L->bufs.end()) continue;
    int err = 0, r2 = read_err_flag(L, "enc_err", &err);
    if (r2 == HIMGCU_OK && err && (rc == HIMGCU_OK || failed_image >= 0)) {
      const int code = enc_err_status(ctx, err);
      if (failed_image >= 0) ctx->err += " (image " + std::to_string(failed_image) + ")";
      return code;
    }
  }
  return rc;
}

int himgcu_encode_status(himgcu_ctx *ctx) {
  if (!ctx) return HIMGCU_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  if (ctx->bufs.find("enc_err") == ctx->bufs.end()) return HIMGCU_OK;
  int err = 0;
  const int rc = read_err_flag(ctx, "enc_err", &err);  // synchronises the stream, clears the flag
  if (rc) return rc;
  return enc_err_status(ctx, err);
}

int himgcu_decode_batch_host(himgcu_ctx *ctx, const uint8_t *himg, const uint64_t *offsets, const uint32_t *sizes,
                             int n, int w, int h, int nch, int flags, uint8_t *pixels_out, int32_t *status) {
  if (!ctx || !himg || !offsets || !sizes || !pixels_out || !status || n < 0) return fail(ctx, HIMGCU_ERR_ARG, "bad argument");
  if (!shape_ok(w, h, nch)) return fail(ctx, HIMGCU_ERR_UNSUPPORTED, "unsupported shape %dx%dx%d", w, h, nch);
  CK(cudaSetDevice(ctx->device));
  int rc = ensure_pipeline(ctx);
  if (rc) return rc;
  const Geom g = make_geom(w, h, nch, nch);
  int sub = (int)std::max<size_t>(1, std::min<size_t>((size_t)std::max(n, 1), ctx->host_sub_bytes / (2 * g.out_img_bytes)));
  sub = std::min(sub, 65535);
  const int K = (n + sub - 1) / sub;
  // contiguous host range of every sub-batch
  std::vector<uint64_t> lo(K), hi(K);
  size_t max_range = 0;
  for (int k = 0; k < K; ++k) {
    const int i0 = k * sub, m = std::min(sub, n - i0);
    lo[k] = offsets[i0];
    hi[k] = 0;
    for (int i = 0; i < m; ++i) {
      lo[k] = std::min<uint64_t>(lo[k], offsets[i0 + i]);
      hi[k] = std::max<uint64_t>(hi[k], offsets[i0 + i] + sizes[i0 + i]);
    }
    max_range = std::max<size_t>(max_range, (size_t)(hi[k] - lo[k]));
  }
  int S = 1;
  if ((rc = prepare_lanes(ctx, K, &S))) return rc;
  uint8_t *d_px[himgcu_ctx::kMaxLanes], *d_in[himgcu_ctx::kMaxLanes];
  unsigned long long *d_off[himgcu_ctx::kMaxLanes];
  uint32_t *d_sz[himgcu_ctx::kMaxLanes];
  int *d_status[himgcu_ctx::kMaxLanes];
  for (int b = 0; b < S; ++b) {
    const std::string sfx = std::to_string(b);
    ENSURE(("hbd_px" + sfx).c_str(), (size_t)sub * g.out_img_bytes, d_px[b]);
    ENSURE(("hbd_in" + sfx).c_str(), max_range + 64, d_in[b]);
    ENSURE(("hbd_off" + sfx).c_str(), (size_t)sub * sizeof(unsigned long long), d_off[b]);
    ENSURE(("hbd_sz" + sfx).c_str(), (size_t)sub * sizeof(uint32_t), d_sz[b]);
    ENSURE(("hbd_status" + sfx).c_str(), (size_t)sub * sizeof(int), d_status[b]);
  }
  // offsets / sizes / status travel through pinned staging: a copy from or to the caller's pageable
  // arrays would block the issuing thread on every sub-batch and serialise the pipeline
  rc = ensure_pinned(ctx, (size_t)n * (sizeof(unsigned long long) + sizeof(uint32_t) + sizeof(int32_t)));
  if (rc) return rc;
  unsigned long long *rel = reinterpret_cast<unsigned long long *>(ctx->pinned);  // stays valid until the end
  uint32_t *p_sz = reinterpret_cast<uint32_t *>(rel + n);
  int32_t *p_status = reinterpret_cast<int32_t *>(p_sz + n);
  memcpy(p_sz, sizes, (size_t)n * sizeof(uint32_t));
  cudaStream_t s_in = ctx->in_stream, s_out = ctx->out_stream;
  for (int b = 0; b < S; ++b) CK(cudaStreamSynchronize(lane_of(ctx, b)->stream));
  PipeTrace trace("dec");
  rc = run_pipeline(
      ctx, K, S, s_in, s_out,
      [&](int k, int b) -> int {
        const int i0 = k * sub, m = std::min(sub, n - i0);
        for (int i = 0; i < m; ++i) rel[i0 + i] = offsets[i0 + i] - lo[k];
        trace.mark(k, 0, s_in);
        CK(cudaMemcpyAsync(d_in[b], himg + lo[k], (size_t)(hi[k] - lo[k]), cudaMemcpyHostToDevice, s_in));
        CK(cudaMemcpyAsync(d_off[b], rel + i0, (size_t)m * sizeof(unsigned long long), cudaMemcpyHostToDevice, s_in));
        CK(cudaMemcpyAsync(d_sz[b], p_sz + i0, (size_t)m * sizeof(uint32_t), cudaMemcpyHostToDevice, s_in));
        trace.mark(k, 1, s_in);
        return HIMGCU_OK;
      },
      [&](int k, int b, himgcu_ctx *L) -> int {
        const int m = std::min(sub, n - k * sub);
        trace.launched(k);
        int r = decode_device(L, d_in[b], d_off[b], d_sz[b], m, g, flags, d_px[b], d_status[b]);
        if (r) return r;
        trace.mark(k, 2, L->stream);
        return HIMGCU_OK;
      },
      [&](int k, int b) -> int {
        const int i0 = k * sub, m = std::min(sub, n - i0);
        CK(cudaMemcpyAsync(p_status + i0, d_status[b], (size_t)m * sizeof(int), cudaMemcpyDeviceToHost, s_out));
        CK(cudaMemcpyAsync(pixels_out + (size_t)i0 * g.out_img_bytes, d_px[b], (size_t)m * g.out_img_bytes, cudaMemcpyDeviceToHost, s_out));
        trace.mark(k, 3, s_out);
        return HIMGCU_OK;
      });
  if (rc) return rc;
  memcpy(status, p_status, (size_t)n * sizeof(int32_t));
  return HIMGCU_OK;
}

// ---- stage-level entry points ------------------------------------------------------------------

int himgcu_stage_lowres(himgcu_ctx *ctx, const uint8_t *d_pixels, int n, int w, int h, int pixel_stride, int nch,
                        int use_ycbcr, uint8_t *d_L) {
  if (!ctx || !d_pixels || !d_L || n < 1 || !shape_ok(w, h, nch) || pixel_stride < nch) return fail(ctx, HIMGCU_ERR_ARG, "bad argument");
  CK(cudaSetDevice(ctx->device));
  return stage_lowres(ctx, d_pixels, n, make_geom(w, h, nch, pixel_stride), use_ycbcr && nch >= 3, d_L);
}

int himgcu_stage_lres_encode(himgcu_ctx *ctx, const uint8_t *d_L, int n, int w, int h, int nch, int quality,
                             uint8_t *d_lres) {
  if (!ctx || !d_L || !d_lres || n < 1 || !shape_ok(w, h, nch)) return fail(ctx, HIMGCU_ERR_ARG, "bad argument");
  CK(cudaSetDevice(ctx->device));
  EncodeTables t;
  BuildEncodeTables(quality, false, &t);
  return stage_lres_encode(ctx, d_L, n, make_geom(w, h, nch, nch), t, d_lres);
}

int himgcu_stage_forward(himgcu_ctx *ctx, const uint8_t *d_pixels, const uint8_t *d_L, int n, int w, int h,
                         int pixel_stride, int nch, int quality, int use_ycbcr, uint8_t *d_planes) {
  if (!ctx || !d_pixels || !d_L || !d_planes || n < 1 || !shape_ok(w, h, nch) || pixel_stride < nch)
    return fail(ctx, HIMGCU_ERR_ARG, "bad argument");
  CK(cudaSetDevice(ctx->device));
  EncodeTables t;
  BuildEncodeTables(quality, use_ycbcr && nch >= 3, &t);
  return stage_forward(ctx, d_pixels, d_L, n, make_geom(w, h, nch, pixel_stride), t, d_planes);
}

int himgcu_stage_huff_compress(himgcu_ctx *ctx, const uint8_t *d_in, size_t in_stride, int n, int in_size,
                               int block_size, uint8_t *d_out, size_t out_stride, uint32_t *d_sizes) {
  if (!ctx || !d_in || !d_out || !d_sizes || n < 1 || in_size < 1) return fail(ctx, HIMGCU_ERR_ARG, "bad argument");
  if (block_size < 1) block_size = in_size;
  if (in_size % block_size) return fail(ctx, HIMGCU_ERR_ARG, "in_size is not a multiple of block_size");
  if (in_size / block_size > 65535) return fail(ctx, HIMGCU_ERR_UNSUPPORTED, "too many segments");
  if (block_size > kMaxSegBytes) return fail(ctx, HIMGCU_ERR_UNSUPPORTED, "segment larger than 2^26 bytes");
  CK(cudaSetDevice(ctx->device));
  HuffChunkArgs ch;
  ch.d_in = d_in;
  ch.hg = HuffGeom{block_size, in_size / block_size, (unsigned long long)in_stride, 1, block_size};
  ch.tag = "stage";
  ch.size_patch = -1;
  return huff_encode_items(ctx, n, &ch, 1, false, d_out, out_stride, d_sizes);
}

int himgcu_stage_huff_uncompress(himgcu_ctx *ctx, const uint8_t *d_in, size_t in_stride, const uint32_t *d_in_sizes,
                                 int n, int out_size, int block_size, int flags, uint8_t *d_out, size_t out_stride,
                                 int32_t *d_status) {
  if (!ctx || !d_in || !d_in_sizes || !d_out || !d_status || n < 1 || out_size < 1) return fail(ctx, HIMGCU_ERR_ARG, "bad argument");
  const int lenient = (flags & HIMGCU_LENIENT) ? 1 : 0;
  const bool whole = block_size < 1;  // Uncompress() vs UncompressBlock()
  const int seg = whole ? out_size : block_size;
  if (out_size % seg || (seg & 3)) return fail(ctx, HIMGCU_ERR_ARG, "segment size must divide out_size and be a multiple of 4");
  if (out_stride & 3) return fail(ctx, HIMGCU_ERR_ARG, "out_stride must be a multiple of 4");
  if (seg > kMaxSegBytes) return fail(ctx, HIMGCU_ERR_UNSUPPORTED, "segment larger than 2^26 bytes");
  const int nseg = out_size / seg;
  CK(cudaSetDevice(ctx->device));
  ChunkDesc *d_cd;
  DecTree *d_tree;
  SegRef *d_seg;
  ENSURE("stage_cd", (size_t)n * sizeof(ChunkDesc), d_cd);
  ENSURE("stage_dtree", (size_t)n * sizeof(DecTree), d_tree);
  ENSURE("stage_dseg", (size_t)n * nseg * sizeof(SegRef), d_seg);
  const unsigned nb = (unsigned)((n + 127) / 128);
  LAUNCH("k_dec_make_desc", k_dec_make_desc, nb, 128, 0, (unsigned long long)in_stride, d_in_sizes, n, d_cd, d_status);
  LAUNCH("k_dec_tree", k_dec_tree, dim3(n, 1), kDecTreeThreads, 0, d_in, d_cd, d_cd, lenient, d_tree, d_tree, d_status);
  LAUNCH("k_dec_segtab", k_dec_segtab, nb, 128, 0, d_in, d_cd, d_tree, n, nseg, seg, whole ? 0 : 1, lenient, d_seg,
         d_status);
  const int team = decode_team((long long)n * nseg, seg, nseg == 1 ? kParLresThreads : kParFresThreads);
  if (nseg == 1 && use_decode_cluster(n, seg) && !ctx->force_generic) {
    bool clustered = false;
    int rc = launch_stream_cluster(ctx, "k_dec_stream", n, d_in, d_cd, d_tree, d_seg, seg, d_out, (unsigned long long)out_stride,
                                   d_status, &clustered);
    if (rc || clustered) return rc;
  }
  return launch_stream_segments(ctx, "k_dec_stream", team, n, d_in, d_cd, d_tree, d_seg, nseg, seg, d_out,
                                (unsigned long long)out_stride, d_status);
}

int himgcu_stage_lres_decode(himgcu_ctx *ctx, const uint8_t *d_lres, size_t lres_stride, int n, int w, int h, int nch,
                             const int16_t *unmap, uint8_t *d_R) {
  if (!ctx || !d_lres || !unmap || !d_R || n < 1 || !shape_ok(w, h, nch)) return fail(ctx, HIMGCU_ERR_ARG, "bad argument");
  CK(cudaSetDevice(ctx->device));
  Geom g = make_geom(w, h, nch, nch);
  g.lres_stride = lres_stride;
  LowResTables *d_tabs;
  int rc = upload_lowres_tables(ctx, nullptr, unmap, &d_tabs);
  if (rc) return rc;
  const long long nmb = (long long)n * g.nch * g.mrows * g.mcols;
  const unsigned blocks = (unsigned)((nmb + kLresWarps * 2 - 1) / (kLresWarps * 2));
  LAUNCH("k_lres_dpcm_dec", (k_lres_dpcm<false>), blocks, kLresWarps * 32, 0, (const uint8_t *)nullptr,
         const_cast<uint8_t *>(d_lres), d_R, g, n, (const uint8_t *)nullptr, d_tabs->unmap, (unsigned long long)0);
  return HIMGCU_OK;
}

int himgcu_stage_inverse(himgcu_ctx *ctx, const uint8_t *d_planes, const uint8_t *d_R, int n, int w, int h, int nch,
                         int use_ycbcr, const uint8_t *shift_luma, const uint8_t *shift_chroma, const int16_t *unmap,
                         uint8_t *d_pixels) {
  if (!ctx || !d_planes || !d_R || !shift_luma || !shift_chroma || !unmap || !d_pixels || n < 1 || !shape_ok(w, h, nch))
    return fail(ctx, HIMGCU_ERR_ARG, "bad argument");
  CK(cudaSetDevice(ctx->device));
  DecTables t;
  memset(&t, 0, sizeof(t));
  memcpy(t.full_unmap, unmap, sizeof(t.full_unmap));
  memcpy(t.shift[0], shift_luma, 64);
  memcpy(t.shift[1], shift_chroma, 64);
  t.ycbcr = (use_ycbcr && nch >= 3) ? 1 : 0;
  DecTables *d_t;
  ENSURE("stage_dectabs", sizeof(DecTables), d_t);
  CK(cudaMemcpyAsync(d_t, &t, sizeof(t), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return stage_inverse(ctx, d_planes, d_R, n, make_geom(w, h, nch, nch), d_t, 0, d_pixels);
}

// ---- profiling ---------------------------------------------------------------------------------

int himgcu_profile_enable(himgcu_ctx *ctx, int on) {
  if (!ctx) return HIMGCU_ERR_ARG;
  ctx->profile = on != 0;
  return HIMGCU_OK;
}

int himgcu_profile_reset(himgcu_ctx *ctx) {
  if (!ctx) return HIMGCU_ERR_ARG;
  cudaStreamSynchronize(ctx->stream);
  resolve_profile(ctx);
  ctx->prof.clear();
  ctx->prof_names.clear();
  return HIMGCU_OK;
}

int himgcu_profile_count(himgcu_ctx *ctx) {
  if (!ctx) return 0;
  cudaStreamSynchronize(ctx->stream);
  resolve_profile(ctx);
  return (int)ctx->prof_names.size();
}

int himgcu_profile_get(himgcu_ctx *ctx, int index, const char **name, double *total_ms, int *launches) {
  if (!ctx || index < 0 || index >= (int)ctx->prof_names.size()) return HIMGCU_ERR_ARG;
  const std::string &k = ctx->prof_names[index];
  if (name) *name = k.c_str();
  if (total_ms) *total_ms = ctx->prof[k].first;
  if (launches) *launches = ctx->prof[k].second;
  return HIMGCU_OK;
}

uint64_t himgcu_launch_count(himgcu_ctx *ctx) { return ctx ? ctx->launches : 0; }

int himgcu_set_option(himgcu_ctx *ctx, const char *name, long long value) {
  if (!ctx || !name) return HIMGCU_ERR_ARG;
  if (!strcmp(name, "force_generic")) ctx->force_generic = value != 0;
  else if (!strcmp(name, "xform_variant")) ctx->xform_variant = (int)value;
  else if (!strcmp(name, "max_workspace_bytes")) ctx->max_workspace = (size_t)value;
  else if (!strcmp(name, "item_lists")) ctx->item_lists = value != 0;
  else if (!strcmp(name, "huff_warp_teams")) ctx->huff_warp_teams = (int)std::max<long long>(0, std::min<long long>(value, 2));
  else if (!strcmp(name, "host_sub_batch_bytes")) ctx->host_sub_bytes = (size_t)std::max<long long>(value, 1 << 20);
  else if (!strcmp(name, "host_lanes")) ctx->host_lanes = (int)std::max<long long>(1, std::min<long long>(value, himgcu_ctx::kMaxLanes));
  else return fail(ctx, HIMGCU_ERR_ARG, "unknown option %s", name);
  return HIMGCU_OK;
}

}  // extern "C"
