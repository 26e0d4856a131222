/* ORACLE -- TEST INFRASTRUCTURE ONLY (see himg_oracle.h).
 *
 * Plain-C restatement of the HIMG codec hot path, written from the behavioural specification
 * in SURVEY.md Appendix A.  Every function cites the reference file:line it restates.  The
 * formulations are deliberately the "specification" ones (e.g. the stale-padding-bit RULE
 * rather than an emulation of the reference's uncleared scratch buffer, a generated scan
 * order, two independent Huffman tree constructions that must agree) so that agreement with
 * the compiled reference actually validates the rules the CUDA kernels implement.
 *
 * All arithmetic is integer with C semantics: >> on negatives is arithmetic, / truncates.
 */
#include "himg_oracle.h"

#include <stdlib.h>
#include <string.h>

/* ======================================================================================== */
/* Synthetic generator + hash (SURVEY Appendix B)                                            */
/* ======================================================================================== */

static uint32_t mix32(uint32_t h) {
  h ^= h >> 16;
  h *= 0x7feb352dU;
  h ^= h >> 15;
  h *= 0x846ca68bU;
  h ^= h >> 16;
  return h;
}

static uint32_t tri(uint32_t t, uint32_t period) {
  uint32_t m = t % period;
  return m < period / 2 ? m : period - 1 - m;
}

void ho_synth_image(uint8_t *out, int w, int h, int nch, uint32_t seed, uint32_t amp) {
  for (uint32_t y = 0; y < (uint32_t)h; ++y)
    for (uint32_t x = 0; x < (uint32_t)w; ++x)
      for (uint32_t k = 0; k < (uint32_t)nch; ++k) {
        int v = 40 + (int)tri(x * (k + 2) + y, 256) + (int)tri(y * 3 + k * 40, 128) +
                ((((x >> 6) + (y >> 6)) & 1) ? 24 : 0);
        if (amp) {
          uint32_t r = mix32(seed * 0x9E3779B9U + ((y * (uint32_t)w + x) * 4U + k));
          v += (int)(r % (2 * amp + 1)) - (int)amp;
        }
        out[((size_t)y * w + x) * nch + k] = (uint8_t)(v < 0 ? 0 : (v > 255 ? 255 : v));
      }
}

uint64_t ho_fnv1a64(const uint8_t *p, size_t n) {
  uint64_t h = 1469598103934665603ULL;
  for (size_t i = 0; i < n; ++i) h = (h ^ p[i]) * 1099511628211ULL;
  return h;
}

/* ======================================================================================== */
/* Tables                                                                                    */
/* ======================================================================================== */

/* quantize.cpp:19-40 -- base tables (data). */
static const uint8_t kLumaBase[64] = {
    16, 11, 10, 16, 24,  40,  51,  61,  12, 12, 14, 19, 26,  58,  60,  55,
    14, 13, 16, 24, 40,  57,  69,  56,  14, 17, 22, 29, 51,  87,  80,  62,
    18, 22, 37, 56, 68,  109, 103, 77,  24, 35, 55, 64, 81,  104, 113, 92,
    49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99};
static const uint8_t kChromaBase[64] = {
    17,  18,  24,  47,  100, 110, 115, 120, 18,  21,  26,  66,  100, 110, 118, 121,
    24,  26,  56,  100, 100, 110, 120, 122, 47,  66,  100, 100, 100, 110, 120, 123,
    100, 100, 100, 100, 100, 110, 120, 124, 110, 110, 110, 110, 110, 110, 110, 123,
    120, 120, 120, 120, 120, 110, 100, 122, 124, 124, 126, 126, 125, 123, 122, 105};

typedef struct {
  int q, s;
} QS;
/* quantize.cpp:55-65 */
static const QS kShiftScale[] = {{0, 65535}, {10, 32512}, {20, 13568}, {30, 5120}, {40, 2560},
                                 {50, 1024}, {60, 768},   {80, 256},   {100, 0}};
/* mapper.cpp:38-47 */
static const QS kLowScale[] = {{0, 120}, {5, 90}, {10, 70}, {20, 40}, {30, 32}, {40, 26}, {50, 20}, {100, 16}};

/* quantize.cpp:72-92 == mapper.cpp:75-97: piece-wise linear, truncating division. */
static int lerp_table(int q, const QS *t, int n) {
  int i = 0;
  while (i < n - 1 && t[i + 1].q <= q) ++i;
  if (i >= n - 1) return t[n - 1].s;
  int den = t[i + 1].q - t[i].q;
  return t[i].s + ((t[i + 1].s - t[i].s) * (q - t[i].q) + (den >> 1)) / den;
}

/* quantize.cpp:94-102 */
static int nearest_log2(unsigned x) {
  int y = 0, r = 0;
  while (x > 1) {
    ++y;
    r = (int)(x & 1u);
    x >>= 1;
  }
  return y + r;
}

/* quantize.cpp:104-114.  `quality` is a uint8_t in the reference (Quantize::InitForQuality). */
void ho_shift_table(int quality, int chroma, uint8_t out[64]) {
  const uint8_t *base = chroma ? kChromaBase : kLumaBase;
  int scale = lerp_table((int)(uint8_t)quality, kShiftScale, 9);
  for (int i = 0; i < 64; ++i) {
    unsigned c = (unsigned)(((int)base[i] * scale + 512) >> 10) & 0xffffu;
    int s = nearest_log2(c);
    out[i] = (uint8_t)(s > 15 ? 15 : s);
  }
}

/* mapper.cpp:19-36 (data): identity up to 65, then a hand-tuned ramp. */
static const uint8_t kLowTail[62] = {67,  68,  70,  71,  73,  74,  76,  78,  79,  81,  83,  85,  87,
                                     89,  91,  93,  95,  97,  99,  102, 104, 106, 109, 111, 114, 117,
                                     119, 122, 125, 128, 131, 134, 137, 140, 143, 146, 150, 153, 156,
                                     160, 164, 167, 171, 175, 178, 182, 186, 190, 195, 199, 203, 207,
                                     212, 216, 221, 226, 230, 235, 240, 245, 250, 255};
static int low_base(int i) { return i <= 65 ? i : kLowTail[i - 66]; }

/* mapper.cpp:193-211 */
void ho_lowres_map_table(int quality, uint16_t t[128]) {
  int scale = lerp_table(quality, kLowScale, 8);
  for (int i = 0; i < 128; ++i) {
    int idx = (int)(int16_t)((i * (int16_t)scale + 8) >> 4);
    if (idx > 127) idx = 127;
    t[i] = (uint16_t)low_base(idx);
  }
}

/* mapper.cpp:54-71 (data): identity up to 49, then roughly geometric. */
static const uint16_t kFullTail[78] = {
    51,   52,   54,   57,   59,   62,   65,   68,   72,   76,   81,   86,   92,   98,   105,  113,
    121,  130,  140,  151,  163,  176,  190,  205,  221,  239,  259,  280,  303,  327,  354,  382,
    413,  446,  482,  520,  561,  605,  653,  703,  757,  815,  876,  942,  1013, 1087, 1167, 1252,
    1342, 1438, 1540, 1649, 1764, 1885, 2015, 2151, 2296, 2450, 2612, 2783, 2965, 3156, 3358, 3571,
    3796, 4032, 4282, 4545, 4821, 5112, 5418, 5740, 6078, 6433, 6806, 7198, 7608, 8039};

/* mapper.cpp:213-223 */
void ho_fullres_map_table(uint16_t t[128]) {
  for (int i = 0; i < 128; ++i) t[i] = (uint16_t)(i <= 49 ? i : kFullTail[i - 50]);
}

/* mapper.cpp:159-182.  Ties go up; anything >= t[126] becomes 127; non-zero never maps to 0. */
int ho_map_to_8bit(const uint16_t t[128], int x) {
  if (x == 0) return 0;
  int a = x < 0 ? -x : x;
  int m = 1;
  while (m < 126) {
    if (a < (int)(int16_t)t[m + 1]) {
      if (a - (int)(int16_t)t[m] < (int)(int16_t)t[m + 1] - a) --m;
      break;
    }
    ++m;
  }
  if (m < 127) ++m;
  return x > 0 ? m : (256 - m) & 0xff;
}

/* mapper.cpp:99-125, :184-191 */
int ho_mapfun_serialize(const uint16_t t[128], uint8_t *out) {
  int n1 = 0;
  while (n1 < 127 && (int16_t)t[n1 + 1] < 256) ++n1;
  int p = 0;
  out[p++] = (uint8_t)n1;
  for (int i = 1; i <= 127; ++i) {
    if (i <= n1) {
      out[p++] = (uint8_t)t[i];
    } else {
      out[p++] = (uint8_t)(t[i] & 255);
      out[p++] = (uint8_t)(t[i] >> 8);
    }
  }
  return p;
}

/* mapper.cpp:127-157.  unmap[] is indexed by the raw code byte: unmap[c] = t[(int8)c]. */
int ho_mapfun_parse(const uint8_t *in, int size, int16_t unmap[256]) {
  if (size < 1) return 0;
  int n1 = in[0];
  if (1 + n1 + 2 * (127 - n1) != size) return 0;
  int16_t t[128];
  int p = 1;
  t[0] = 0;
  for (int i = 1; i <= 127; ++i) {
    if (i <= n1) {
      t[i] = (int16_t)in[p++];
    } else {
      t[i] = (int16_t)(uint16_t)(in[p] | (in[p + 1] << 8));
      p += 2;
    }
  }
  for (int c = 0; c < 128; ++c) unmap[c] = t[c];
  for (int k = 1; k <= 127; ++k) unmap[256 - k] = (int16_t)(-t[k]);
  unmap[128] = unmap[129]; /* t[-128] = t[-127] */
  return 1;
}

/* Encoder-side unmap table straight from a magnitude table. */
static void unmap_from_table(const uint16_t t[128], int16_t unmap[256]) {
  for (int c = 0; c < 128; ++c) unmap[c] = (int16_t)t[c];
  for (int k = 1; k <= 127; ++k) unmap[256 - k] = (int16_t)(-(int16_t)t[k]);
  unmap[128] = unmap[129];
}

/* common.cpp:13-22 -- generated instead of tabulated: L-shaped shells, odd shells run down the
 * new column then left along the new row, even shells run right along the new row then up. */
static void scan_order(uint8_t lut[64]) {
  int n = 0;
  for (int k = 0; k < 8; ++k) {
    if (k & 1) {
      for (int r = 0; r <= k; ++r) lut[n++] = (uint8_t)(r * 8 + k);
      for (int c = k - 1; c >= 0; --c) lut[n++] = (uint8_t)(k * 8 + c);
    } else {
      for (int c = 0; c <= k; ++c) lut[n++] = (uint8_t)(k * 8 + c);
      for (int r = k - 1; r >= 0; --r) lut[n++] = (uint8_t)(r * 8 + k);
    }
  }
}

/* ======================================================================================== */
/* Colour mapping                                                                            */
/* ======================================================================================== */

static int clamp255(int x) { return x < 0 ? 0 : (x > 255 ? 255 : x); }

/* ycbcr.cpp:24-52 */
void ho_rgb_to_ycbcr(const uint8_t *in, uint8_t *out, int w, int h, int stride, int nch) {
  size_t n = (size_t)w * h;
  for (size_t i = 0; i < n; ++i, in += stride, out += stride) {
    int r = in[0], g = in[1], b = in[2];
    out[0] = (uint8_t)((r + 2 * g + b + 2) >> 2);
    out[1] = (uint8_t)((b - g + 256) >> 1);
    out[2] = (uint8_t)((r - g + 256) >> 1);
    for (int c = 3; c < nch; ++c) out[c] = in[c];
  }
}

/* ycbcr.cpp:54-82 */
void ho_ycbcr_to_rgb(uint8_t *buf, int w, int h, int nch) {
  size_t n = (size_t)w * h;
  for (size_t i = 0; i < n; ++i, buf += nch) {
    int y = buf[0], cb = 2 * buf[1] - 255, cr = 2 * buf[2] - 255;
    int g = y - ((cb + cr + 2) >> 2);
    buf[0] = (uint8_t)clamp255(g + cr);
    buf[1] = (uint8_t)clamp255(g);
    buf[2] = (uint8_t)clamp255(g + cb);
  }
}

/* ======================================================================================== */
/* Low-res image                                                                             */
/* ======================================================================================== */

/* downsampled.cpp:67-114 */
void ho_lowres_sample(const uint8_t *pix, int stride, int w, int h, uint8_t *L) {
  int rows = (h + 7) >> 3, cols = (w + 7) >> 3;
  uint8_t *avg = (uint8_t *)malloc((size_t)rows * cols);
  for (int v = 0; v < rows; ++v) {
    int y0 = 8 * v - 3 < 0 ? 0 : 8 * v - 3, y1 = 8 * v + 4 > h - 1 ? h - 1 : 8 * v + 4;
    for (int u = 0; u < cols; ++u) {
      int x0 = 8 * u - 3 < 0 ? 0 : 8 * u - 3, x1 = 8 * u + 4 > w - 1 ? w - 1 : 8 * u + 4;
      unsigned sum = 0;
      for (int y = y0; y <= y1; ++y)
        for (int x = x0; x <= x1; ++x) sum += pix[((size_t)y * w + x) * stride];
      sum &= 0xffffu; /* uint16_t accumulator in the reference (never wraps: <= 64*255) */
      int n = (x1 - x0 + 1) * (y1 - y0 + 1);
      avg[v * cols + u] = (uint8_t)(((int)sum + (n >> 1)) / n);
    }
  }
  for (int v = 0; v < rows; ++v) {
    int vp = v > 0 ? v - 1 : 0;
    for (int u = 0; u < cols; ++u) {
      int up = u > 0 ? u - 1 : 0;
      int a1 = (avg[vp * cols + up] + 15 * avg[vp * cols + u] + 8) >> 4;
      int a2 = (avg[v * cols + up] + 15 * avg[v * cols + u] + 8) >> 4;
      L[v * cols + u] = (uint8_t)((a1 + 15 * a2 + 8) >> 4);
    }
  }
  free(avg);
}

/* downsampled.cpp:171-175 */
int ho_lowres_channel_size(int rows, int cols) {
  return ((rows + 15) / 16) * ((cols + 15) / 16) + rows * cols;
}

/* downsampled.cpp:41-60.  Anything but 1..4 selects the mixed predictor. */
static int predict(int s1, int s2, int s3, int p) {
  switch (p) {
    case 1: return s2;
    case 2: return s3;
    case 3: return (s2 + s3 + 1) >> 1;
    case 4: return clamp255(s2 + s3 - s1);
    default: return clamp255((3 * (s2 + s3) - 2 * s1 + 2) >> 2);
  }
}

/* Neighbour rule shared by encoder and decoder (downsampled.cpp:204-219, :272-283, :345-357). */
static void neighbours(const uint8_t *X, int cols, int v, int u, int dv, int du, int *s1, int *s2,
                       int *s3) {
  if (du > 0 && dv > 0) {
    *s1 = X[(v - 1) * cols + u - 1];
    *s2 = X[(v - 1) * cols + u];
    *s3 = X[v * cols + u - 1];
  } else if (du > 0) {
    *s1 = *s2 = *s3 = X[v * cols + u - 1];
  } else if (dv > 0) {
    *s1 = *s2 = *s3 = X[(v - 1) * cols + u];
  } else {
    *s1 = *s2 = *s3 = 128;
  }
}

/* downsampled.cpp:177-316.  out = sel[mrows*mcols] ++ deltas in macroblock-major order. */
void ho_lowres_encode(const uint8_t *L, int rows, int cols, const uint16_t lt[128], uint8_t *out) {
  int mrows = (rows + 15) / 16, mcols = (cols + 15) / 16;
  int16_t unmap[256];
  unmap_from_table(lt, unmap);
  uint8_t *sel = out;
  uint8_t *delta = out + mrows * mcols;
  uint8_t *R = (uint8_t *)calloc((size_t)rows * cols, 1);
  for (int mv = 0; mv < mrows; ++mv)
    for (int mu = 0; mu < mcols; ++mu) {
      long err[5] = {0, 0, 0, 0, 0};
      for (int dv = 0; dv < 16 && mv * 16 + dv < rows; ++dv)
        for (int du = 0; du < 16 && mu * 16 + du < cols; ++du) {
          int v = mv * 16 + dv, u = mu * 16 + du, s1, s2, s3;
          neighbours(L, cols, v, u, dv, du, &s1, &s2, &s3);
          for (int p = 0; p < 5; ++p) {
            int d = L[v * cols + u] - predict(s1, s2, s3, p);
            err[p] += d * d;
          }
        }
      int best = 0;
      for (int p = 1; p < 5; ++p)
        if (err[p] < err[best]) best = p;
      sel[mv * mcols + mu] = (uint8_t)(best - 2);
    }
  for (int mv = 0; mv < mrows; ++mv)
    for (int mu = 0; mu < mcols; ++mu) {
      /* The byte is widened to int BEFORE adding 2, so 254/255 become 256/257 and fall to the
       * default predictor (downsampled.cpp:37-39) -- SURVEY A.4-4. */
      int p = (int)sel[mv * mcols + mu] + 2;
      for (int dv = 0; dv < 16 && mv * 16 + dv < rows; ++dv)
        for (int du = 0; du < 16 && mu * 16 + du < cols; ++du) {
          int v = mv * 16 + dv, u = mu * 16 + du, s1, s2, s3;
          neighbours(R, cols, v, u, dv, du, &s1, &s2, &s3);
          int pr = predict(s1, s2, s3, p);
          int d8 = ho_map_to_8bit(lt, L[v * cols + u] - pr);
          R[v * cols + u] = (uint8_t)clamp255(pr + unmap[d8]);
          *delta++ = (uint8_t)d8;
        }
    }
  free(R);
}

/* downsampled.cpp:318-382 */
void ho_lowres_decode(const uint8_t *in, int rows, int cols, const int16_t unmap[256], uint8_t *R) {
  int mrows = (rows + 15) / 16, mcols = (cols + 15) / 16;
  const uint8_t *sel = in;
  const uint8_t *delta = in + mrows * mcols;
  for (int mv = 0; mv < mrows; ++mv)
    for (int mu = 0; mu < mcols; ++mu) {
      int p = (int)sel[mv * mcols + mu] + 2;
      for (int dv = 0; dv < 16 && mv * 16 + dv < rows; ++dv)
        for (int du = 0; du < 16 && mu * 16 + du < cols; ++du) {
          int v = mv * 16 + dv, u = mu * 16 + du, s1, s2, s3;
          neighbours(R, cols, v, u, dv, du, &s1, &s2, &s3);
          int pr = predict(s1, s2, s3, p);
          int x = (int16_t)(pr + unmap[*delta++]);
          R[v * cols + u] = (uint8_t)clamp255(x);
        }
    }
}

static void nine(int a, int b, int t[9]) {
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

/* downsampled.cpp:116-169 */
void ho_lowres_block(const uint8_t *X, int rows, int cols, int u, int v, int16_t out[64]) {
  int v2 = v + 1 < rows ? v + 1 : rows - 1, u2 = u + 1 < cols ? u + 1 : cols - 1;
  int left[9], right[9], row[9];
  nine(X[v * cols + u], X[v2 * cols + u], left);
  nine(X[v * cols + u2], X[v2 * cols + u2], right);
  for (int y = 0; y < 8; ++y) {
    nine(left[y], right[y], row);
    for (int x = 0; x < 8; ++x) out[y * 8 + x] = (int16_t)row[x];
  }
}

/* ======================================================================================== */
/* Transform + quantisation                                                                  */
/* ======================================================================================== */

/* hadamard.cpp:18-44: sequency-ordered 8-point WHT. */
static void wht8(const int *x, int *o) {
  int a0 = x[0] + x[4], a1 = x[1] + x[5], a2 = x[2] + x[6], a3 = x[3] + x[7];
  int a4 = x[0] - x[4], a5 = x[1] - x[5], a6 = x[2] - x[6], a7 = x[3] - x[7];
  int b0 = a0 + a2, b1 = a1 + a3, b2 = a0 - a2, b3 = a1 - a3;
  int b4 = a4 + a6, b5 = a5 + a7, b6 = a4 - a6, b7 = a5 - a7;
  o[0] = b0 + b1;
  o[1] = b4 + b5;
  o[2] = b6 + b7;
  o[3] = b2 + b3;
  o[4] = b2 - b3;
  o[5] = b6 - b7;
  o[6] = b4 - b5;
  o[7] = b0 - b1;
}

/* hadamard.cpp:78-88 (int16 storage between passes) */
void ho_wht_forward(const int16_t in[64], int16_t out[64]) {
  int x[8], o[8];
  int16_t tmp[64];
  for (int r = 0; r < 8; ++r) {
    for (int i = 0; i < 8; ++i) x[i] = in[r * 8 + i];
    wht8(x, o);
    for (int i = 0; i < 8; ++i) tmp[r * 8 + i] = (int16_t)o[i];
  }
  for (int c = 0; c < 8; ++c) {
    for (int i = 0; i < 8; ++i) x[i] = tmp[i * 8 + c];
    wht8(x, o);
    for (int i = 0; i < 8; ++i) out[i * 8 + c] = (int16_t)o[i];
  }
}

/* hadamard.cpp:90-103: int32 butterflies, floor >>3 after EACH pass, int16 storage. */
void ho_wht_inverse(const int16_t in[64], int16_t out[64]) {
  int x[8], o[8];
  int16_t tmp[64];
  for (int r = 0; r < 8; ++r) {
    for (int i = 0; i < 8; ++i) x[i] = in[r * 8 + i];
    wht8(x, o);
    for (int i = 0; i < 8; ++i) tmp[r * 8 + i] = (int16_t)(o[i] >> 3);
  }
  for (int c = 0; c < 8; ++c) {
    for (int i = 0; i < 8; ++i) x[i] = tmp[i * 8 + c];
    wht8(x, o);
    for (int i = 0; i < 8; ++i) out[i * 8 + c] = (int16_t)(o[i] >> 3);
  }
}

/* encoder.cpp:26-52 -- edge replication quirk: columns past the edge repeat the row's last valid
 * pixel; rows past the edge are filled with the single last value written. */
static void extract_block(const uint8_t *cm, int w, int h, int stride, int c, int u, int v,
                          int16_t out[64]) {
  int bw = w - 8 * u < 8 ? w - 8 * u : 8, bh = h - 8 * v < 8 ? h - 8 * v : 8;
  int last = 0;
  for (int y = 0; y < 8; ++y)
    for (int x = 0; x < 8; ++x) {
      if (y < bh && x < bw) last = cm[((size_t)(8 * v + y) * w + 8 * u + x) * stride + c];
      out[y * 8 + x] = (int16_t)last;
    }
}

/* encoder.cpp:258-335 + quantize.cpp:127-151 */
void ho_fullres_planes(const uint8_t *cm, int w, int h, int stride, int nch, int ycbcr,
                       const uint8_t *L, const uint8_t shift_luma[64],
                       const uint8_t shift_chroma[64], const uint16_t ft[128], uint8_t *planes) {
  int rows = (h + 7) >> 3, cols = (w + 7) >> 3;
  uint8_t scan[64];
  scan_order(scan);
  size_t idx = 0;
  for (int v = 0; v < rows; ++v)
    for (int c = 0; c < nch; ++c) {
      const uint8_t *sh = (ycbcr && (c == 1 || c == 2)) ? shift_chroma : shift_luma;
      for (int u = 0; u < cols; ++u) {
        int16_t blk[64], lo[64], tr[64];
        uint8_t q[64];
        extract_block(cm, w, h, stride, c, u, v, blk);
        ho_lowres_block(L + (size_t)c * rows * cols, rows, cols, u, v, lo);
        for (int i = 0; i < 64; ++i) blk[i] = (int16_t)(blk[i] - lo[i]);
        ho_wht_forward(blk, tr);
        for (int j = 0; j < 64; ++j) {
          int s = sh[j], r = s ? 1 << (s - 1) : 0, x = tr[j];
          int m = x < 0 ? -((-x + r) >> s) : (x + r) >> s;
          q[j] = (uint8_t)ho_map_to_8bit(ft, (int16_t)m);
        }
        for (int i = 0; i < 64; ++i) planes[idx + (size_t)i * cols + u] = q[scan[i]];
      }
      idx += (size_t)cols * 64;
    }
}

/* decoder.cpp:331-426 + quantize.cpp:153-165.  Width not a multiple of 8 is undefined in the
 * reference (decoder.cpp:63-72); here it is DEFINED as cropping. */
void ho_fullres_restore(const uint8_t *planes, int w, int h, int nch, int ycbcr, const uint8_t *R,
                        const uint8_t shift_luma[64], const uint8_t shift_chroma[64],
                        const int16_t unmap[256], uint8_t *out) {
  int rows = (h + 7) >> 3, cols = (w + 7) >> 3;
  uint8_t scan[64];
  scan_order(scan);
  size_t idx = 0;
  for (int v = 0; v < rows; ++v) {
    int bh = h - 8 * v < 8 ? h - 8 * v : 8;
    for (int c = 0; c < nch; ++c) {
      const uint8_t *sh = (ycbcr && nch >= 3 && (c == 1 || c == 2)) ? shift_chroma : shift_luma;
      for (int u = 0; u < cols; ++u) {
        int bw = w - 8 * u < 8 ? w - 8 * u : 8;
        int16_t co[64], px[64], lo[64];
        for (int i = 0; i < 64; ++i) {
          int j = scan[i];
          int val = unmap[planes[idx + (size_t)i * cols + u]];
          co[j] = (int16_t)(val * (1 << sh[j]));
        }
        ho_wht_inverse(co, px);
        ho_lowres_block(R + (size_t)c * rows * cols, rows, cols, u, v, lo);
        for (int y = 0; y < bh; ++y)
          for (int x = 0; x < bw; ++x) {
            int16_t s = (int16_t)(px[y * 8 + x] + lo[y * 8 + x]);
            out[((size_t)(8 * v + y) * w + 8 * u + x) * nch + c] = (uint8_t)clamp255(s);
          }
      }
      idx += (size_t)cols * 64;
    }
    if (ycbcr && nch >= 3) ho_ycbcr_to_rgb(out + (size_t)8 * v * w * nch, w, bh, nch);
  }
}

/* ======================================================================================== */
/* RLE + Huffman                                                                             */
/* ======================================================================================== */

enum { SYM_Z2 = 256, SYM_Z6 = 257, SYM_Z22 = 258, SYM_Z278 = 259, SYM_Z16662 = 260, MAX_RUN = 16662 };

/* Token at position k of a segment: returns symbol, sets *adv (bytes consumed), *extra / *nextra.
 * huffman_enc.cpp:105-141 == :296-336. */
static int next_token(const uint8_t *seg, size_t k, size_t seg_size, int *adv, uint32_t *extra, int *nextra) {
  *extra = 0;
  *nextra = 0;
  if (seg[k] != 0) {
    *adv = 1;
    return seg[k];
  }
  int z = 1;
  while (z < MAX_RUN && k + z < seg_size && seg[k + z] == 0) ++z;
  *adv = z;
  if (z == 1) return 0;
  if (z == 2) return SYM_Z2;
  if (z <= 6) {
    *extra = (uint32_t)(z - 3);
    *nextra = 2;
    return SYM_Z6;
  }
  if (z <= 22) {
    *extra = (uint32_t)(z - 7);
    *nextra = 4;
    return SYM_Z22;
  }
  if (z <= 278) {
    *extra = (uint32_t)(z - 23);
    *nextra = 8;
    return SYM_Z278;
  }
  *extra = (uint32_t)(z - 279);
  *nextra = 14;
  return SYM_Z16662;
}

/* huffman_enc.cpp:98-144 */
void ho_huff_histogram(const uint8_t *in, size_t in_size, size_t block_size, uint32_t hist[HO_NUM_SYMBOLS]) {
  memset(hist, 0, sizeof(uint32_t) * HO_NUM_SYMBOLS);
  if (block_size < 1) block_size = in_size;
  for (size_t base = 0; base < in_size; base += block_size)
    for (size_t k = 0; k < block_size;) {
      int adv, nx;
      uint32_t ex;
      hist[next_token(in + base, k, block_size, &adv, &ex, &nx)]++;
      k += adv;
    }
}

typedef struct {
  uint8_t *p;
  size_t bit;
} BitW;

static void put_bits(BitW *w, uint32_t x, int n) { /* LSB first, huffman_enc.cpp:31-53 */
  for (int i = 0; i < n; ++i, ++w->bit)
    if ((x >> i) & 1u) w->p[w->bit >> 3] |= (uint8_t)(1u << (w->bit & 7));
}

typedef struct {
  int a, b, sym;
  uint64_t count;
} TNode;

/* Direct statement of huffman_enc.cpp:183-227: repeatedly join the two minima under the order
 * (count ascending, node index DEscending); child_a = lightest. Returns root index, -1 if empty. */
static int build_tree_direct(const uint32_t hist[HO_NUM_SYMBOLS], TNode *nd, int *nleaves) {
  int n = 0;
  for (int s = 0; s < HO_NUM_SYMBOLS; ++s)
    if (hist[s]) {
      nd[n].a = nd[n].b = -1;
      nd[n].sym = s;
      nd[n].count = hist[s];
      ++n;
    }
  *nleaves = n;
  if (n == 0) return -1;
  int next = n, left = n, root = 0;
  while (left > 1) {
    int n1 = -1, n2 = -1;
    for (int k = 0; k < next; ++k) {
      if (!nd[k].count) continue;
      if (n1 < 0 || nd[k].count <= nd[n1].count) {
        n2 = n1;
        n1 = k;
      } else if (n2 < 0 || nd[k].count <= nd[n2].count) {
        n2 = k;
      }
    }
    root = next++;
    nd[root].a = n1;
    nd[root].b = n2;
    nd[root].sym = -1;
    nd[root].count = nd[n1].count + nd[n2].count;
    nd[n1].count = nd[n2].count = 0;
    --left;
  }
  return root;
}

/* Same tree in O(n log n): leaves sorted by (count asc, index desc) feed a queue; internal nodes
 * are created with non-decreasing counts, so they form groups of equal count that are consumed
 * front group first and NEWEST first inside a group (higher node index wins ties).  An internal
 * node beats a leaf of equal count (internal indices are larger).  This is the algorithm the
 * device kernel runs; the test-suite requires it to match build_tree_direct exactly. */
static int build_tree_fast(const uint32_t hist[HO_NUM_SYMBOLS], TNode *nd, int *nleaves) {
  int n = 0;
  for (int s = 0; s < HO_NUM_SYMBOLS; ++s)
    if (hist[s]) {
      nd[n].a = nd[n].b = -1;
      nd[n].sym = s;
      nd[n].count = hist[s];
      ++n;
    }
  *nleaves = n;
  if (n == 0) return -1;
  if (n == 1) return 0;
  int lq[HO_NUM_SYMBOLS]; /* rank sort: keys are unique */
  for (int i = 0; i < n; ++i) {
    int rank = 0;
    for (int j = 0; j < n; ++j)
      if (nd[j].count < nd[i].count || (nd[j].count == nd[i].count && j > i)) ++rank;
    lq[rank] = i;
  }
  int ist[HO_NUM_SYMBOLS];                       /* internal node ids, creation order */
  int g_start[HO_NUM_SYMBOLS], g_top[HO_NUM_SYMBOLS]; /* group ranges inside ist[] */
  uint64_t g_count[HO_NUM_SYMBOLS];
  int ist_n = 0, gfront = 0, glast = -1, lp = 0, next = n, root = 0;
  for (int merge = 0; merge < n - 1; ++merge) {
    int pick[2];
    for (int k = 0; k < 2; ++k) {
      /* drop exhausted front groups */
      while (gfront < glast && g_top[gfront] == g_start[gfront]) ++gfront;
      int have_int = glast >= 0 && gfront <= glast &&
                     (gfront == glast ? ist_n > g_start[glast] : g_top[gfront] > g_start[gfront]);
      int take_int = have_int && (lp >= n || g_count[gfront] <= nd[lq[lp]].count);
      if (take_int) {
        if (gfront == glast) {
          pick[k] = ist[--ist_n];
        } else {
          pick[k] = ist[--g_top[gfront]];
        }
      } else {
        pick[k] = lq[lp++];
      }
    }
    root = next++;
    nd[root].a = pick[0];
    nd[root].b = pick[1];
    nd[root].sym = -1;
    nd[root].count = nd[pick[0]].count + nd[pick[1]].count;
    /* push: joins the last group if it has the same count, else opens a new group at the tail */
    if (glast >= 0 && ist_n > g_start[glast] && g_count[glast] == nd[root].count) {
      ist[ist_n++] = root;
    } else if (glast >= 0 && ist_n == g_start[glast]) {
      g_count[glast] = nd[root].count; /* empty last group is reused */
      ist[ist_n++] = root;
    } else {
      if (glast >= 0) g_top[glast] = ist_n;
      ++glast;
      g_start[glast] = ist_n;
      g_count[glast] = nd[root].count;
      ist[ist_n++] = root;
    }
  }
  return root;
}

/* huffman_enc.cpp:148-180, :229-237: pre-order serialisation, leaf = 1 + 9-bit symbol, branch = 0;
 * code bit k (LSB first) is the branch taken at depth k (child_b => 1). */
int ho_huff_tree(const uint32_t hist[HO_NUM_SYMBOLS], int fast, uint32_t code[HO_NUM_SYMBOLS],
                 uint8_t len[HO_NUM_SYMBOLS], uint8_t *tree_bytes) {
  TNode nd[HO_MAX_NODES];
  int nleaves;
  int root = fast ? build_tree_fast(hist, nd, &nleaves) : build_tree_direct(hist, nd, &nleaves);
  memset(code, 0, sizeof(uint32_t) * HO_NUM_SYMBOLS);
  memset(len, 0, HO_NUM_SYMBOLS);
  memset(tree_bytes, 0, 360);
  if (root < 0) return 0;
  BitW w = {tree_bytes, 0};
  int st_node[HO_MAX_NODES], st_bits[HO_MAX_NODES], sp = 0;
  uint32_t st_code[HO_MAX_NODES];
  st_node[0] = root;
  st_bits[0] = nleaves == 1 ? 1 : 0;
  st_code[0] = 0;
  sp = 1;
  while (sp) {
    --sp;
    int k = st_node[sp], bits = st_bits[sp];
    uint32_t c = st_code[sp];
    if (nd[k].sym >= 0) {
      put_bits(&w, 1, 1);
      put_bits(&w, (uint32_t)nd[k].sym, 9);
      if (bits > 32) return -1; /* undefined in the reference (1 << bits on uint32) */
      code[nd[k].sym] = c;
      len[nd[k].sym] = (uint8_t)bits;
    } else {
      put_bits(&w, 0, 1);
      st_node[sp] = nd[k].b; /* visited second */
      st_bits[sp] = bits + 1;
      st_code[sp] = bits < 32 ? c + (1u << bits) : c;
      ++sp;
      st_node[sp] = nd[k].a;
      st_bits[sp] = bits + 1;
      st_code[sp] = c;
      ++sp;
    }
  }
  return (int)w.bit;
}

/* huffman_enc.cpp:242-244 */
size_t ho_huff_max_size(size_t n) { return n + ((2 + 9) * HO_NUM_SYMBOLS + 7) / 8; }

/* huffman_enc.cpp:246-363.  Returns the packed size, 0 for the reference's "nothing to do"
 * cases, -1 if `out_cap` is too small. */
long long ho_huff_compress(uint8_t *out, size_t out_cap, const uint8_t *in, size_t in_size, size_t block_size) {
  if (in_size < 1) return 0;
  if (block_size < 1) block_size = in_size;
  int framed = block_size < in_size;
  if (in_size % block_size != 0) return 0;
  uint32_t hist[HO_NUM_SYMBOLS], code[HO_NUM_SYMBOLS];
  uint8_t len[HO_NUM_SYMBOLS];
  ho_huff_histogram(in, in_size, block_size, hist);
  uint8_t tree[360];
  int tree_bits = ho_huff_tree(hist, 0, code, len, tree);
  if (tree_bits < 0) return 0;
  size_t pos = (size_t)(tree_bits + 7) / 8;

  size_t nseg = in_size / block_size;
  size_t *seg_bits = (size_t *)malloc(sizeof(size_t) * nseg);
  size_t *seg_pos = (size_t *)malloc(sizeof(size_t) * nseg);
  /* pass 1: bit length of every segment -> layout */
  size_t total = pos;
  for (size_t b = 0; b < nseg; ++b) {
    const uint8_t *seg = in + b * block_size;
    size_t bits = 0;
    for (size_t k = 0; k < block_size;) {
      int adv, nx;
      uint32_t ex;
      int s = next_token(seg, k, block_size, &adv, &ex, &nx);
      bits += (size_t)len[s] + nx;
      k += adv;
    }
    seg_bits[b] = bits;
    size_t size = (bits + 7) / 8;
    total += size + (framed ? (size <= 0x7fff ? 2 : 4) : 0);
  }
  if (total > out_cap) {
    free(seg_bits);
    free(seg_pos);
    return -1;
  }
  memcpy(out, tree, pos);
  /* pass 2: emit */
  for (size_t b = 0; b < nseg; ++b) {
    const uint8_t *seg = in + b * block_size;
    size_t bits = seg_bits[b], size = (bits + 7) / 8;
    if (framed) { /* :340-352 */
      if (size <= 0x7fff) {
        out[pos++] = (uint8_t)(size & 255);
        out[pos++] = (uint8_t)(size >> 8);
      } else {
        size_t lo = (size & 0x7fff) | 0x8000, hi = size >> 15;
        out[pos++] = (uint8_t)(lo & 255);
        out[pos++] = (uint8_t)(lo >> 8);
        out[pos++] = (uint8_t)(hi & 255);
        out[pos++] = (uint8_t)(hi >> 8);
      }
    }
    memset(out + pos, 0, size);
    BitW w = {out + pos, 0};
    for (size_t k = 0; k < block_size;) {
      int adv, nx;
      uint32_t ex;
      int s = next_token(seg, k, block_size, &adv, &ex, &nx);
      put_bits(&w, code[s], len[s]);
      put_bits(&w, ex, nx);
      k += adv;
    }
    seg_pos[b] = pos;
    /* Stale padding bits (SURVEY A.3 step 5): each padding bit position p of this segment takes
     * the value that the most recent earlier segment with more than p bits WROTE there. */
    for (size_t p = bits; p < 8 * size; ++p)
      for (size_t e = b; e-- > 0;)
        if (seg_bits[e] > p) {
          if ((out[seg_pos[e] + (p >> 3)] >> (p & 7)) & 1u) out[pos + (p >> 3)] |= (uint8_t)(1u << (p & 7));
          break;
        }
    pos += size;
  }
  free(seg_bits);
  free(seg_pos);
  return (long long)pos;
}

typedef struct {
  const uint8_t *p;
  size_t bit, nbits;
  int fail;
} BitR;

static int get_bit(BitR *r) {
  if (r->bit >= r->nbits) {
    r->fail = 1;
    return 0;
  }
  int b = (r->p[r->bit >> 3] >> (r->bit & 7)) & 1;
  ++r->bit;
  return b;
}

static uint32_t get_bits(BitR *r, int n) {
  if (r->bit + (size_t)n > r->nbits) {
    r->fail = 1;
    return 0;
  }
  uint32_t x = 0;
  for (int i = 0; i < n; ++i) x |= (uint32_t)get_bit(r) << i;
  return x;
}

typedef struct {
  int a[HO_MAX_NODES], b[HO_MAX_NODES], sym[HO_MAX_NODES];
  int n;
} DTree;

/* huffman_dec.cpp:152-213 (iterative, with an effective node limit). Returns 1 ok. */
static int parse_tree(BitR *r, DTree *t) {
  /* explicit stack of "slot to fill": encoded as node*2 + which (0 = a, 1 = b); -1 = root */
  int stack[HO_MAX_NODES + 2], sp = 0;
  t->n = 0;
  stack[sp++] = -1;
  while (sp) {
    int slot = stack[--sp];
    if (t->n >= HO_MAX_NODES) return 0;
    int k = t->n++;
    t->a[k] = t->b[k] = -1;
    t->sym[k] = -1;
    if (slot >= 0) {
      if (slot & 1) t->b[slot >> 1] = k;
      else t->a[slot >> 1] = k;
    }
    int leaf = get_bit(r);
    if (r->fail) return 0;
    if (leaf) {
      t->sym[k] = (int)get_bits(r, 9);
      if (r->fail) return 0;
    } else {
      stack[sp++] = k * 2 + 1; /* b after a */
      stack[sp++] = k * 2;
    }
  }
  return 1;
}

/* huffman_dec.cpp:274-418.  Fully checked (hostile streams are rejected, never over-read). */
static int decode_stream(const DTree *t, const uint8_t *p, size_t size, uint8_t *out, size_t out_size,
                         int strict) {
  BitR r = {p, 0, size * 8, 0};
  size_t n = 0;
  while (n < out_size) {
    int k = 0;
    while (t->sym[k] < 0) {
      k = get_bit(&r) ? t->b[k] : t->a[k];
      if (r.fail) return 0;
    }
    /* Single-leaf tree: the encoder spends 1 bit per token (huffman_enc.cpp:233-237) but the
     * reference decoder consumes none (huffman_dec.cpp:178-188) and then fails its end check;
     * lenient mode consumes the bit. */
    if (t->n == 1 && !strict) {
      get_bit(&r);
      if (r.fail) return 0;
    }
    int s = t->sym[k];
    if (s <= 255) {
      out[n++] = (uint8_t)s;
      continue;
    }
    size_t z;
    switch (s) {
      case SYM_Z2: z = 2; break;
      case SYM_Z6: z = get_bits(&r, 2) + 3; break;
      case SYM_Z22: z = get_bits(&r, 4) + 7; break;
      case SYM_Z278: z = get_bits(&r, 8) + 23; break;
      case SYM_Z16662: z = get_bits(&r, 14) + 279; break;
      default: return 0;
    }
    if (r.fail || n + z > out_size) return 0;
    memset(out + n, 0, z);
    n += z;
  }
  /* BitStream::AtTheEnd, huffman_dec.cpp:140-145: the read position must lie in the last byte
   * (or exactly at the end). */
  return size == 0 ? r.bit == 0 : (r.bit > 8 * (size - 1) && r.bit <= 8 * size);
}

int ho_huff_uncompress(const uint8_t *in, size_t in_size, size_t block_size, int block_no, uint8_t *out,
                       size_t out_size, int strict, size_t unpacked_total) {
  BitR r = {in, 0, in_size * 8, 0};
  DTree *t = (DTree *)malloc(sizeof(DTree));
  int ok = 0;
  if (!parse_tree(&r, t)) goto done;
  size_t pos = (r.bit + 7) / 8;
  size_t bs = block_size > 0 ? block_size : in_size;
  /* huffman_dec.cpp:215-219: the reference compares the UNPACKED block size with the PACKED
   * chunk size (SURVEY A.4-6); lenient mode uses what the encoder did. */
  int framed = strict ? bs < in_size : (block_size > 0 && block_size < unpacked_total);
  /* lenient: a chunk with a single segment is unframed (huffman_enc.cpp:254-256) */
  if (!strict && !framed && block_no == 0) block_no = -1;
  if (block_no < 0) {
    if (framed) goto done;
    if (pos == in_size) { /* :278-279 */
      ok = out_size == 0;
      goto done;
    }
    ok = decode_stream(t, in + pos, in_size - pos, out, out_size, strict);
    goto done;
  }
  if (!framed) goto done; /* UncompressBlock refuses, huffman_dec.cpp:265 */
  for (int b = 0;; ++b) { /* :233-248 */
    if (pos == in_size) goto done; /* table ended before block_no */
    if (pos + 2 > in_size) goto done;
    size_t sz = in[pos] | ((size_t)in[pos + 1] << 8);
    pos += 2;
    if (sz & 0x8000) {
      if (pos + 2 > in_size) goto done;
      sz = (sz & 0x7fff) | ((size_t)(in[pos] | (in[pos + 1] << 8)) << 15);
      pos += 2;
    }
    if (pos + sz > in_size) goto done;
    if (b == block_no) {
      ok = decode_stream(t, in + pos, sz, out, out_size, strict);
      goto done;
    }
    pos += sz;
  }
done:
  free(t);
  return ok;
}

/* ======================================================================================== */
/* Whole codec                                                                               */
/* ======================================================================================== */

static void put_u32(uint8_t *p, uint32_t x) {
  p[0] = (uint8_t)x;
  p[1] = (uint8_t)(x >> 8);
  p[2] = (uint8_t)(x >> 16);
  p[3] = (uint8_t)(x >> 24);
}

static uint32_t get_u32(const uint8_t *p) {
  return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}

static size_t put_chunk_hdr(uint8_t *out, size_t pos, const char *fourcc, uint32_t size) {
  memcpy(out + pos, fourcc, 4);
  put_u32(out + pos + 4, size);
  return pos + 8;
}

size_t ho_encode_bound(int w, int h, int nch) {
  size_t rows = (size_t)(h + 7) >> 3, cols = (size_t)(w + 7) >> 3;
  size_t lres = (size_t)ho_lowres_channel_size((int)rows, (int)cols) * nch;
  size_t fres = rows * cols * 64 * nch;
  return 12 + 19 + 136 + 8 + 72 + 188 + 8 + ho_huff_max_size(lres) + ho_huff_max_size(fres);
}

/* encoder.cpp:59-109 (container layout: SURVEY A.1) */
long long ho_encode(const uint8_t *data, int w, int h, int pixel_stride, int nch, int quality,
                    int use_ycbcr, uint8_t *out, size_t out_cap) {
  int ycbcr = use_ycbcr && nch >= 3;
  int rows = (h + 7) >> 3, cols = (w + 7) >> 3;
  size_t npix = (size_t)w * h;
  uint8_t *cm = (uint8_t *)malloc(npix * pixel_stride);
  if (ycbcr) ho_rgb_to_ycbcr(data, cm, w, h, pixel_stride, nch);
  else memcpy(cm, data, npix * pixel_stride);

  uint16_t lt[128], ft[128];
  uint8_t sl[64], sc[64];
  ho_lowres_map_table(quality, lt);
  ho_fullres_map_table(ft);
  ho_shift_table(quality, 0, sl);
  ho_shift_table(quality, 1, sc);

  int chsz = ho_lowres_channel_size(rows, cols);
  uint8_t *L = (uint8_t *)malloc((size_t)rows * cols * nch);
  uint8_t *lres = (uint8_t *)malloc((size_t)chsz * nch);
  for (int c = 0; c < nch; ++c) {
    ho_lowres_sample(cm + c, pixel_stride, w, h, L + (size_t)c * rows * cols);
    ho_lowres_encode(L + (size_t)c * rows * cols, rows, cols, lt, lres + (size_t)c * chsz);
  }
  size_t fres_n = (size_t)rows * cols * 64 * nch;
  uint8_t *planes = (uint8_t *)malloc(fres_n);
  ho_fullres_planes(cm, w, h, pixel_stride, nch, ycbcr, L, sl, sc, ft, planes);

  size_t tmp_cap = 2 * ((size_t)chsz * nch + fres_n) + 8192;
  uint8_t *tmp = (uint8_t *)calloc(tmp_cap, 1);
  size_t pos = 0;
  memcpy(tmp, "RIFF\0\0\0\0HIMG", 12);
  pos = 12;
  pos = put_chunk_hdr(tmp, pos, "FRMT", 11);
  tmp[pos++] = 1;
  put_u32(tmp + pos, (uint32_t)w);
  put_u32(tmp + pos + 4, (uint32_t)h);
  pos += 8;
  tmp[pos++] = (uint8_t)nch;
  tmp[pos++] = (uint8_t)(ycbcr ? 1 : 0);
  {
    uint8_t mf[256];
    int n = ho_mapfun_serialize(lt, mf);
    pos = put_chunk_hdr(tmp, pos, "LMAP", (uint32_t)n);
    memcpy(tmp + pos, mf, (size_t)n);
    pos += (size_t)n;
  }
  {
    long long n = ho_huff_compress(tmp + pos + 8, tmp_cap - pos - 8, lres, (size_t)chsz * nch, 0);
    if (n < 0) n = 0;
    pos = put_chunk_hdr(tmp, pos, "LRES", (uint32_t)n) + (size_t)n;
  }
  {
    int n = ycbcr ? 64 : 32;
    pos = put_chunk_hdr(tmp, pos, "QCFG", (uint32_t)n);
    for (int i = 0; i < 32; ++i) tmp[pos++] = (uint8_t)((sl[2 * i] << 4) | sl[2 * i + 1]);
    if (ycbcr)
      for (int i = 0; i < 32; ++i) tmp[pos++] = (uint8_t)((sc[2 * i] << 4) | sc[2 * i + 1]);
  }
  {
    uint8_t mf[256];
    int n = ho_mapfun_serialize(ft, mf);
    pos = put_chunk_hdr(tmp, pos, "FMAP", (uint32_t)n);
    memcpy(tmp + pos, mf, (size_t)n);
    pos += (size_t)n;
  }
  {
    long long n = ho_huff_compress(tmp + pos + 8, tmp_cap - pos - 8 - 512, planes, fres_n, (size_t)cols * nch * 64);
    if (n < 0) n = 0;
    pos = put_chunk_hdr(tmp, pos, "FRES", (uint32_t)n) + (size_t)n;
  }
  put_u32(tmp + 4, (uint32_t)(pos - 8));
  long long ret = pos <= out_cap ? (long long)pos : -1;
  if (ret > 0) memcpy(out, tmp, pos);
  free(tmp);
  free(planes);
  free(lres);
  free(L);
  free(cm);
  return ret;
}

/* decoder.cpp:428-461 */
static int find_chunk(const uint8_t *p, size_t size, size_t *idx, const char *fourcc, size_t *chunk_size) {
  for (;;) {
    if (*idx + 8 > size) return 0;
    uint32_t cc = get_u32(p + *idx);
    int32_t sz = (int32_t)get_u32(p + *idx + 4);
    *idx += 8;
    if (sz < 0 || *idx + (size_t)sz > size) return 0;
    if (cc == get_u32((const uint8_t *)fourcc)) {
      *chunk_size = (size_t)sz;
      return 1;
    }
    *idx += sz;
  }
}

/* decoder.cpp:87-138 */
int ho_decode(const uint8_t *packed, size_t size, int strict, uint8_t *out, size_t out_cap, int *w,
              int *h, int *nch) {
  if (size < 12 || memcmp(packed, "RIFF", 4) || memcmp(packed + 8, "HIMG", 4)) return 0;
  if ((long long)(int32_t)get_u32(packed + 4) + 8 != (long long)size) return 0;
  size_t idx = 12, cs;
  if (!find_chunk(packed, size, &idx, "FRMT", &cs) || cs < 11) return 0;
  const uint8_t *c = packed + idx;
  idx += cs;
  if (c[0] != 1) return 0;
  int W = (int32_t)get_u32(c + 1), H = (int32_t)get_u32(c + 5), N = c[9], ycbcr = c[10] != 0;
  if (W < 1 || H < 1 || N < 1) return 0; /* undefined in the reference */
  *w = W;
  *h = H;
  *nch = N;
  int has_chroma = ycbcr && N >= 3;
  int rows = (H + 7) >> 3, cols = (W + 7) >> 3;

  int16_t lun[256], fun[256];
  if (!find_chunk(packed, size, &idx, "LMAP", &cs) || !ho_mapfun_parse(packed + idx, cs, lun)) return 0;
  idx += cs;

  if (!find_chunk(packed, size, &idx, "LRES", &cs)) return 0;
  int chsz = ho_lowres_channel_size(rows, cols);
  uint8_t *lres = (uint8_t *)malloc((size_t)chsz * N);
  uint8_t *R = (uint8_t *)malloc((size_t)rows * cols * N);
  uint8_t *planes = NULL;
  int ret = 0;
  if (!ho_huff_uncompress(packed + idx, cs, 0, -1, lres, (size_t)chsz * N, strict, (size_t)chsz * N)) goto done;
  idx += cs;
  for (int k = 0; k < N; ++k)
    ho_lowres_decode(lres + (size_t)k * chsz, rows, cols, lun, R + (size_t)k * rows * cols);

  uint8_t sl[64], sc[64];
  memset(sc, 0, 64);
  if (!find_chunk(packed, size, &idx, "QCFG", &cs) || cs != (has_chroma ? 64 : 32)) goto done;
  for (int i = 0; i < 32; ++i) {
    sl[2 * i] = packed[idx + i] >> 4;
    sl[2 * i + 1] = packed[idx + i] & 15;
    if (has_chroma) {
      sc[2 * i] = packed[idx + 32 + i] >> 4;
      sc[2 * i + 1] = packed[idx + 32 + i] & 15;
    }
  }
  idx += cs;
  if (!find_chunk(packed, size, &idx, "FMAP", &cs) || !ho_mapfun_parse(packed + idx, cs, fun)) goto done;
  idx += cs;

  if (!find_chunk(packed, size, &idx, "FRES", &cs)) goto done;
  if ((size_t)W * H * N > out_cap) {
    ret = -1;
    goto done;
  }
  size_t seg = (size_t)cols * 64 * N;
  planes = (uint8_t *)malloc(seg * rows);
  for (int v = 0; v < rows; ++v)
    if (!ho_huff_uncompress(packed + idx, cs, seg, v, planes + (size_t)v * seg, seg, strict, seg * rows))
      goto done;
  ho_fullres_restore(planes, W, H, N, ycbcr, R, sl, sc, fun, out);
  ret = 1;
done:
  free(planes);
  free(R);
  free(lres);
  return ret;
}
