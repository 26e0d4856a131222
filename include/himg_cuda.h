/* himg_cuda.h -- C ABI of the B200-native HIMG encode/decode hot path (libhimgcu.so).
 *
 * This is the seam directly beneath the reference's C++ API: the reference has no FFI, its
 * contract is himg::Encoder / himg::Decoder (src/lib/encoder.h:20-64, src/lib/decoder.h:22-67).
 * himg_b200/host/{encoder,decoder}.{h,cpp} keep those two classes verbatim and forward to the
 * entry points below; INTEGRATION.md shows the same two-line change applied to the reference
 * tree.  Plain pointers and sizes only; no C++/torch types; no exceptions cross the boundary.
 *
 * All kernels are hand-written sm_100a CUDA.  There is NO CPU fallback: every entry point
 * returns HIMGCU_ERR_CUDA if no usable device is present.
 *
 * Threading: a context owns one CUDA stream and its device scratch; use one context per host
 * thread (distinct contexts may run concurrently).
 *
 * Accepted shapes (every entry point, including the bounds of the mixed batch calls and the FRMT
 * shape of a stream being decoded; anything else is HIMGCU_ERR_UNSUPPORTED, and encode_bound /
 * lres_size / lres_stride return 0):
 *   1 <= num_channels <= 255;
 *   width * height * num_channels < 2^31 pixel bytes;
 *   ceil(height / 8) <= 65535 block rows;
 *   8 * ceil(width / 8) * num_channels <= 2^23, i.e. a block row of at most 2^26 coefficient bytes
 *   (width * num_channels <= 8 388 608 when width is a multiple of 8).  Such a row codes to fewer
 *   than 2^32 bits, which keeps the entropy coder's bit counts 32-bit.
 * A decoded stream with a coded segment (a framed FRES segment, or a whole unframed chunk) of 2^29
 * bytes or more is rejected.
 */
#ifndef HIMG_CUDA_H_
#define HIMG_CUDA_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct himgcu_ctx himgcu_ctx;

enum {
  HIMGCU_OK = 0,
  HIMGCU_REJECT = 1,          /* stream refused: where himg::Decoder::Decode returns false */
  HIMGCU_ERR_ARG = 2,
  HIMGCU_ERR_CUDA = 3,
  HIMGCU_ERR_CAPACITY = 4,    /* output buffer too small */
  HIMGCU_ERR_UNSUPPORTED = 5  /* e.g. num_channels > 255, Huffman code longer than 32 bits */
};

/* decode flags */
enum {
  HIMGCU_STRICT = 0,  /* mirror the reference decoder's accept/reject decisions (SURVEY A.4-6) */
  HIMGCU_LENIENT = 1  /* also decode the reference encoder's streams its own decoder refuses   */
};

int himgcu_abi_version(void);
int himgcu_device_count(void);

/* Context: device scratch + stream.  `device` is a CUDA ordinal. */
int himgcu_create(int device, himgcu_ctx **out);
void himgcu_destroy(himgcu_ctx *ctx);
/* Run on an externally owned stream (cudaStream_t / CUstream handle, e.g. torch's current
 * stream).  As in the CUDA API, NULL is the legacy default stream.  himgcu_reset_stream goes
 * back to the context's own (non-blocking) stream. */
int himgcu_set_stream(himgcu_ctx *ctx, void *cuda_stream);
int himgcu_reset_stream(himgcu_ctx *ctx);
int himgcu_synchronize(himgcu_ctx *ctx);
const char *himgcu_last_error(himgcu_ctx *ctx);

/* The checksum of SURVEY.md Appendix B over a host buffer (FNV-1a, 64 bit, with the appendix's offset
 * basis 1469598103934665603), exported so that callers can compare bitstreams and images with the
 * recorded reference hashes without a second implementation. */
uint64_t himgcu_fnv1a64(const uint8_t *data, size_t size);

/* Upper bound of an encoded image (same bound as the reference's buffers,
 * huffman_enc.cpp:242-244, encoder.cpp:337-353). */
size_t himgcu_encode_bound(int width, int height, int num_channels);

/* ---- single image, HOST pointers ---------------------------------------------------------
 * Replaces himg::Encoder::Encode (src/lib/encoder.cpp:59-109): `pixels` is interleaved u8,
 * `pixel_stride` bytes between pixels (>= num_channels), rows contiguous, quality 0..100,
 * YCbCr is used iff use_ycbcr && num_channels >= 3.  Copies in, encodes on the device, copies
 * the .himg bytes out; *out_size receives the size. */
int himgcu_encode(himgcu_ctx *ctx, const uint8_t *pixels, int width, int height, int pixel_stride,
                  int num_channels, int quality, int use_ycbcr, uint8_t *out, size_t out_cap,
                  size_t *out_size);

/* Header peek (host only; replaces Decoder::DecodeRIFFStart/DecodeHeader, decoder.cpp:144-200). */
int himgcu_decode_info(const uint8_t *himg, size_t size, int *width, int *height, int *num_channels);

/* Replaces himg::Decoder::Decode (src/lib/decoder.cpp:87-138).  Output is tightly packed
 * [height][width][num_channels].  Returns HIMGCU_REJECT where the reference returns false. */
int himgcu_decode(himgcu_ctx *ctx, const uint8_t *himg, size_t size, int flags, uint8_t *out,
                  size_t out_cap, int *width, int *height, int *num_channels);

/* ---- batch, DEVICE pointers (configs c4/c5: many same-shaped images per GPU) --------------
 * d_pixels: n images, each [height][width][num_channels] tightly packed, image i at
 * d_pixels + i * width*height*num_channels.  Image i's bitstream is written to
 * d_out + i*out_stride and its size to d_sizes[i] (0 and HIMGCU_ERR_CAPACITY if it does not
 * fit in out_stride).  Asynchronous on the context's stream. */
int himgcu_encode_batch(himgcu_ctx *ctx, const uint8_t *d_pixels, int n, int width, int height,
                        int num_channels, int quality, int use_ycbcr, uint8_t *d_out,
                        size_t out_stride, uint32_t *d_sizes);

/* Why an image of an earlier asynchronous himgcu_encode_batch call came out with size 0: synchronises
 * the context's stream and returns (and clears) the encoder's sticky device status -- HIMGCU_OK,
 * HIMGCU_ERR_CAPACITY (did not fit in out_stride), HIMGCU_ERR_UNSUPPORTED (a Huffman code longer than
 * the reference's 32-bit code words, huffman_enc.cpp:179) or HIMGCU_ERR_CUDA (internal mismatch). */
int himgcu_encode_status(himgcu_ctx *ctx);

/* d_himg + d_offsets[i] .. + d_sizes[i] is image i's .himg; every image must have the given
 * shape.  d_status[i] receives HIMGCU_OK / HIMGCU_REJECT per image.  Pixels of image i go to
 * d_pixels_out + i * width*height*num_channels. */
int himgcu_decode_batch(himgcu_ctx *ctx, const uint8_t *d_himg, const uint64_t *d_offsets,
                        const uint32_t *d_sizes, int n, int width, int height, int num_channels,
                        int flags, uint8_t *d_pixels_out, int32_t *d_status);

/* ---- region decode: a rectangle [x, x+rw) x [y, y+rh) of an image ------------------------
 * Pixel (yy, xx) of the output equals pixel (y+yy, x+xx) of himgcu_decode on the same stream with
 * the same flags, for every shape himgcu_decode accepts; the output is [rh][rw][num_channels]
 * tightly packed.  The low-res chunk is decoded in full, but of the FRES chunk only the segment
 * headers up to the rectangle's last 8-pixel block row (at least the first two) and the segments of
 * the block rows the rectangle touches are read.  Everything a whole decode checks is checked where the region reads
 * it: the container, the tables, both trees, the low-res stream, the FRES framing decision, those
 * segment headers and those segments.  So a stream the whole decode accepts is accepted and its
 * pixels are the crop, and a stream the region decode rejects is rejected by the whole decode too;
 * a stream whose corruption lies only in rows below the rectangle, or in segments it does not
 * touch, may decode as a region.
 *
 * Single image, host buffers (as himgcu_decode): HIMGCU_ERR_ARG for an empty rectangle or one
 * outside the image. */
int himgcu_decode_region(himgcu_ctx *ctx, const uint8_t *himg, size_t size, int flags, int x, int y,
                         int rw, int rh, uint8_t *out, size_t out_cap, int *width, int *height,
                         int *num_channels);

/* n same-shaped streams as himgcu_decode_batch, one rectangle size rw x rh for the batch (checked
 * here: HIMGCU_ERR_ARG if empty or larger than the image) and one origin per image in DEVICE memory
 * (d_origins[2i] = x, d_origins[2i+1] = y), so that a caller can draw them on the GPU.  Image i's
 * rectangle goes to d_pixels_out + i*rw*rh*num_channels.  d_status[i]: HIMGCU_OK / HIMGCU_REJECT as
 * in himgcu_decode_batch, or HIMGCU_ERR_ARG if the origin puts the rectangle outside the image (its
 * output is then not written).  Asynchronous on the context's stream. */
int himgcu_decode_batch_region(himgcu_ctx *ctx, const uint8_t *d_himg, const uint64_t *d_offsets,
                               const uint32_t *d_sizes, int n, int width, int height, int num_channels,
                               int flags, const int32_t *d_origins, int rw, int rh,
                               uint8_t *d_pixels_out, int32_t *d_status);

/* n streams of one channel count but each of its own size, as a data loader reads them: d_dims[2i]
 * = width, d_dims[2i+1] = height of image i (DEVICE memory, as d_origins).  max_width x max_height
 * (host) bounds every image and sizes the workspace (HIMGCU_ERR_UNSUPPORTED if it is not a shape
 * himgcu_decode_batch takes).  One rectangle size rw x rh for the batch (HIMGCU_ERR_ARG if empty or
 * larger than the bounds), origins as in himgcu_decode_batch_region; image i's rectangle goes to
 * d_pixels_out + i*rw*rh*num_channels.  Image i's output and status are those of
 * himgcu_decode_region on its stream alone with the same origin and flags, and a batch whose dims
 * are all equal gives what himgcu_decode_batch_region gives.  d_status[i]: HIMGCU_OK; HIMGCU_REJECT
 * where the stream is rejected, including a FRMT shape other than its dims and num_channels; or
 * HIMGCU_ERR_ARG when its dims are < 1 or exceed the bounds, or the origin puts the rectangle
 * outside the image (its output is then not written).  Asynchronous on the context's stream. */
int himgcu_decode_batch_region_mixed(himgcu_ctx *ctx, const uint8_t *d_himg, const uint64_t *d_offsets,
                                     const uint32_t *d_sizes, int n, const int32_t *d_dims, int max_width,
                                     int max_height, int num_channels, int flags, const int32_t *d_origins,
                                     int rw, int rh, uint8_t *d_pixels_out, int32_t *d_status);

/* The encoder's side of the call above: n images of one channel count, each of its own size, in one call.
 * Image i is [h_i][w_i][num_channels], tightly packed at d_pixels + d_pixel_offsets[i] (no alignment
 * required), with d_dims[2i] = w_i and d_dims[2i+1] = h_i; offsets and dims are in DEVICE memory.
 * max_width x max_height (host) bounds every image and sizes the workspace (HIMGCU_ERR_UNSUPPORTED if it
 * is not a shape himgcu_encode_batch takes).  One quality and one use_ycbcr for the batch (YCbCr iff
 * use_ycbcr && num_channels >= 3).  Output as in himgcu_encode_batch: image i's stream at d_out +
 * i*out_stride, its size in d_sizes[i]; asynchronous on the context's stream.  Image i's bytes and size are
 * exactly those of himgcu_encode (or himgcu_encode_batch with n = 1) on that image alone, and a batch whose
 * dims are all equal gives what himgcu_encode_batch gives.  Per image, without effect on the others:
 * dims < 1 or above the bounds give size 0 and nothing is written to its output slot (himgcu_encode_status
 * then reports HIMGCU_ERR_ARG, unless a worse error of the same call outranks it); a stream that does not
 * fit out_stride gives size 0 and HIMGCU_ERR_CAPACITY.  Null pointers and n < 0 are HIMGCU_ERR_ARG; n = 0
 * does nothing.  The transforms are always the generic (one block per thread) kernels, and the option
 * "force_generic" does not change the entropy coder of this call: the first-generation coder it selects
 * elsewhere has no variant for images of their own sizes. */
int himgcu_encode_batch_mixed(himgcu_ctx *ctx, const uint8_t *d_pixels, const uint64_t *d_pixel_offsets,
                              const int32_t *d_dims, int n, int max_width, int max_height, int num_channels,
                              int quality, int use_ycbcr, uint8_t *d_out, size_t out_stride,
                              uint32_t *d_sizes);

/* Whole-image decode of n streams of one channel count, each of its own size: the decoder's side of
 * himgcu_encode_batch_mixed.  Inputs as in himgcu_decode_batch_region_mixed without the rectangle: d_dims[2i]
 * = width, d_dims[2i+1] = height of image i (DEVICE memory), bounded by max_width x max_height (host;
 * HIMGCU_ERR_UNSUPPORTED if it is not a shape himgcu_decode_batch takes).  Image i is written as
 * [h_i][w_i][num_channels], tightly packed, at d_pixels_out + d_pixel_offsets[i] (DEVICE memory, no alignment
 * required); the caller sizes the buffer and keeps the spans from overlapping.  Image i's pixels and status are
 * exactly those of himgcu_decode on its stream alone with the same flags, and a batch whose dims are all equal,
 * with offsets i*w*h*num_channels, gives what himgcu_decode_batch gives.  d_status[i], without effect on the
 * other images: HIMGCU_OK; HIMGCU_REJECT where the stream is rejected, including a FRMT shape other than its dims
 * and num_channels; HIMGCU_ERR_ARG when its dims are < 1 or exceed the bounds (nothing of it is written).  An
 * image with a non-OK status writes nothing outside its own span.  Null pointers and n < 0 are HIMGCU_ERR_ARG;
 * n = 0 does nothing.  Asynchronous on the context's stream.  The inverse transform is always the generic (one
 * block per thread) kernel. */
int himgcu_decode_batch_mixed(himgcu_ctx *ctx, const uint8_t *d_himg, const uint64_t *d_offsets,
                              const uint32_t *d_sizes, int n, const int32_t *d_dims, int max_width,
                              int max_height, int num_channels, int flags,
                              const uint64_t *d_pixel_offsets, uint8_t *d_pixels_out, int32_t *d_status);

/* ---- scaled decode: the image at 1/factor size, averaged inside the inverse transform -----------
 * For factor f in {1, 2, 4, 8} and D = what himgcu_decode gives for the stream with the same flags
 * ([H][W][num_channels]), the output is [ceil(H/f)][ceil(W/f)][num_channels], tightly packed, with
 *     out[y][x][c] = (S + n/2) / n     (integer division)
 * where S is the sum of D[yy][xx][c] over yy in [f*y, min(f*y + f, H)), xx in [f*x, min(f*x + f, W)) and n is the
 * number of pixels of that window inside the image (edge windows are clipped).  The average is taken of the final
 * pixels, after the clamp and the inverse colour map, without a full-size buffer.  Every FRES segment is still
 * entropy-decoded, so statuses and accept/reject decisions are those of the unscaled call; f = 1 gives exactly the
 * unscaled call's output.  Any other factor is HIMGCU_ERR_ARG.  The pixels of an image with a non-OK status are
 * unspecified, but nothing is written outside its own output.
 *
 * Single image, host buffers (as himgcu_decode): width / height / num_channels receive the stream's FULL shape;
 * out_cap is checked against the scaled size (HIMGCU_ERR_CAPACITY if smaller). */
int himgcu_decode_scaled(himgcu_ctx *ctx, const uint8_t *himg, size_t size, int flags, int factor,
                         uint8_t *out, size_t out_cap, int *width, int *height, int *num_channels);

/* himgcu_decode_batch at 1/factor size: image i goes to d_pixels_out + i * ceil(w/f)*ceil(h/f)*num_channels.
 * Arguments, statuses and host-side checks as himgcu_decode_batch, plus HIMGCU_ERR_ARG for a bad factor. */
int himgcu_decode_batch_scaled(himgcu_ctx *ctx, const uint8_t *d_himg, const uint64_t *d_offsets,
                               const uint32_t *d_sizes, int n, int width, int height, int num_channels,
                               int flags, int factor, uint8_t *d_pixels_out, int32_t *d_status);

/* himgcu_decode_batch_mixed at 1/factor size: image i is written as [ceil(h_i/f)][ceil(w_i/f)][num_channels] at
 * d_pixels_out + d_pixel_offsets[i] (no alignment required).  Arguments, per-image statuses (HIMGCU_ERR_ARG for dims
 * out of bounds, HIMGCU_REJECT for a FRMT shape other than the dims) and host-side checks as
 * himgcu_decode_batch_mixed, plus HIMGCU_ERR_ARG for a bad factor.  A batch whose dims are all equal gives what
 * himgcu_decode_batch_scaled gives.  The inverse transform is always the generic kernel. */
int himgcu_decode_batch_mixed_scaled(himgcu_ctx *ctx, const uint8_t *d_himg, const uint64_t *d_offsets,
                                     const uint32_t *d_sizes, int n, const int32_t *d_dims, int max_width,
                                     int max_height, int num_channels, int flags, int factor,
                                     const uint64_t *d_pixel_offsets, uint8_t *d_pixels_out, int32_t *d_status);

/* ---- scaled region decode: a rectangle of the image at 1/factor size ----------------------------
 * The rectangle [x, x+rw) x [y, y+rh) is given in the coordinates of the SCALED image: for f in {1, 2, 4, 8} and
 * S = what himgcu_decode_scaled gives for the stream with the same flags and factor ([ceil(H/f)][ceil(W/f)][nch]),
 *     out[yy][xx][c] = S[y + yy][x + xx][c]
 * and the output is [rh][rw][num_channels], tightly packed (edge windows are clipped as in the scaled calls).  The
 * call reads exactly what himgcu_decode_region reads for the source rectangle (f*x, f*y, min(f*rw, W - f*x),
 * min(f*rh, H - f*y)), and its status is that call's: a stream the whole decode accepts is accepted, and a stream whose
 * corruption lies only below the rectangle's last block row may decode.  f = 1 is exactly the unscaled region call.
 * Any other factor is HIMGCU_ERR_ARG.
 *
 * Single image, host buffers (as himgcu_decode_region): width / height / num_channels receive the stream's FULL
 * shape; HIMGCU_ERR_ARG for an empty rectangle or one outside the scaled image; out_cap is checked against
 * rw*rh*num_channels. */
int himgcu_decode_region_scaled(himgcu_ctx *ctx, const uint8_t *himg, size_t size, int flags, int factor, int x, int y,
                                int rw, int rh, uint8_t *out, size_t out_cap, int *width, int *height,
                                int *num_channels);

/* himgcu_decode_batch_region at 1/factor size: rw x rh is checked here against ceil(width/f) x ceil(height/f)
 * (HIMGCU_ERR_ARG), and d_status[i] is HIMGCU_ERR_ARG if image i's origin puts the rectangle outside the scaled image
 * (nothing of it is written).  Image i's rectangle goes to d_pixels_out + i*rw*rh*num_channels.  Otherwise as
 * himgcu_decode_batch_region, plus HIMGCU_ERR_ARG for a bad factor. */
int himgcu_decode_batch_region_scaled(himgcu_ctx *ctx, const uint8_t *d_himg, const uint64_t *d_offsets,
                                      const uint32_t *d_sizes, int n, int width, int height, int num_channels,
                                      int flags, int factor, const int32_t *d_origins, int rw, int rh,
                                      uint8_t *d_pixels_out, int32_t *d_status);

/* himgcu_decode_batch_region_mixed at 1/factor size: rw x rh is checked against ceil(max_width/f) x
 * ceil(max_height/f), origins against image i's scaled shape.  Image i's rectangle goes to d_pixels_out +
 * i*rw*rh*num_channels.  Per-image statuses (HIMGCU_ERR_ARG for dims out of bounds or an origin outside the scaled
 * image, HIMGCU_REJECT for a FRMT shape other than the dims) as himgcu_decode_batch_region_mixed, plus HIMGCU_ERR_ARG
 * for a bad factor.  A batch whose dims are all equal gives what himgcu_decode_batch_region_scaled gives.  The inverse
 * transform is always the generic kernel. */
int himgcu_decode_batch_region_mixed_scaled(himgcu_ctx *ctx, const uint8_t *d_himg, const uint64_t *d_offsets,
                                            const uint32_t *d_sizes, int n, const int32_t *d_dims, int max_width,
                                            int max_height, int num_channels, int flags, int factor,
                                            const int32_t *d_origins, int rw, int rh, uint8_t *d_pixels_out,
                                            int32_t *d_status);

/* ---- batch, HOST pointers (what a file/stream based caller uses; basis of the e2e figure) ----
 * Same work as the device batch calls with the transfers included: pixels (or bitstreams) are
 * copied host->device in sub-batches, coded, and the results copied back.  Pinned host memory
 * (himgcu_host_alloc) makes the copies asynchronous; pageable memory works but is slower.
 * Encode: image i's bitstream lands at out + offsets[i], offsets[n] = total bytes (each stream
 * is padded to a multiple of 16 bytes; sizes[i] is the exact size). */
void *himgcu_host_alloc(size_t bytes);
void himgcu_host_free(void *p);
int himgcu_encode_batch_host(himgcu_ctx *ctx, const uint8_t *pixels, int n, int width, int height,
                             int num_channels, int quality, int use_ycbcr, uint8_t *out,
                             size_t out_cap, uint64_t *offsets /* [n+1] */, uint32_t *sizes /* [n] */);
int himgcu_decode_batch_host(himgcu_ctx *ctx, const uint8_t *himg, const uint64_t *offsets,
                             const uint32_t *sizes, int n, int width, int height, int num_channels,
                             int flags, uint8_t *pixels_out, int32_t *status /* [n] */);

/* ---- stage-level entry points (DEVICE pointers) -------------------------------------------
 * The pipeline stages above are built from these; they are exported for the parity tests and
 * for per-kernel roofline timing.  n = number of images, shapes as above. */

/* Colour map + 8x8 corner-window average + phase compensation (ycbcr.cpp:24-52,
 * downsampled.cpp:67-114).  d_L: [n][nch][rows][cols] u8. */
int himgcu_stage_lowres(himgcu_ctx *ctx, const uint8_t *d_pixels, int n, int width, int height,
                        int pixel_stride, int num_channels, int use_ycbcr, uint8_t *d_L);

/* Predictor selection + DPCM of the low-res image (downsampled.cpp:177-316).
 * d_lres: [n][lres_stride] with lres_stride = himgcu_lres_stride(...); the first
 * nch*(mb + rows*cols) bytes of each row are the LRES unpacked data. */
size_t himgcu_lres_size(int width, int height, int num_channels);
size_t himgcu_lres_stride(int width, int height, int num_channels);
int himgcu_stage_lres_encode(himgcu_ctx *ctx, const uint8_t *d_L, int n, int width, int height,
                             int num_channels, int quality, uint8_t *d_lres);

/* K-fwd: colour map + low-res subtract + 2-D WHT + shift quantise + 8-bit map + planar scatter
 * (encoder.cpp:258-335).  d_planes: [n][rows][cols*64*nch] = FRES unpacked bytes. */
int himgcu_stage_forward(himgcu_ctx *ctx, const uint8_t *d_pixels, const uint8_t *d_L, int n,
                         int width, int height, int pixel_stride, int num_channels, int quality,
                         int use_ycbcr, uint8_t *d_planes);

/* RLE + Huffman of n equally sized chunks (HuffmanEnc::Compress, huffman_enc.cpp:246-363).
 * Chunk i = d_in + i*in_stride (in_size bytes, block_size as in the reference: 0 = unframed);
 * output i = d_out + i*out_stride, size to d_sizes[i]. */
int himgcu_stage_huff_compress(himgcu_ctx *ctx, const uint8_t *d_in, size_t in_stride, int n,
                               int in_size, int block_size, uint8_t *d_out, size_t out_stride,
                               uint32_t *d_sizes);

/* Inverse (HuffmanDec, huffman_dec.cpp:221-418): d_status[i] = HIMGCU_OK / HIMGCU_REJECT. */
int himgcu_stage_huff_uncompress(himgcu_ctx *ctx, const uint8_t *d_in, size_t in_stride,
                                 const uint32_t *d_in_sizes, int n, int out_size, int block_size,
                                 int flags, uint8_t *d_out, size_t out_stride, int32_t *d_status);

/* DPCM reconstruction (downsampled.cpp:318-382).  unmap: host pointer, int16[256] indexed by the
 * code byte (Mapper::UnmapFrom8Bit, mapper.h:33-35).  d_R: [n][nch][rows][cols]. */
int himgcu_stage_lres_decode(himgcu_ctx *ctx, const uint8_t *d_lres, size_t lres_stride, int n,
                             int width, int height, int num_channels, const int16_t *unmap,
                             uint8_t *d_R);

/* K-inv: gather + dequantise + inverse WHT + low-res add + clamp + inverse colour map
 * (decoder.cpp:331-426).  shift_luma/shift_chroma: host, 64 bytes each; unmap as above. */
int himgcu_stage_inverse(himgcu_ctx *ctx, const uint8_t *d_planes, const uint8_t *d_R, int n,
                         int width, int height, int num_channels, int use_ycbcr,
                         const uint8_t *shift_luma, const uint8_t *shift_chroma,
                         const int16_t *unmap, uint8_t *d_pixels);

/* ---- per-kernel timing (CUDA events on the context's stream) ------------------------------
 * When enabled every kernel launch is bracketed by events; after himgcu_synchronize the
 * accumulated device time per kernel name can be read back.  Used by bench.py for the
 * roofline figure; off by default. */
int himgcu_profile_enable(himgcu_ctx *ctx, int on);
int himgcu_profile_reset(himgcu_ctx *ctx);
int himgcu_profile_count(himgcu_ctx *ctx);
int himgcu_profile_get(himgcu_ctx *ctx, int index, const char **name, double *total_ms, int *launches);
/* Total number of kernels launched through this context since creation. */
uint64_t himgcu_launch_count(himgcu_ctx *ctx);
/* Tuning / test knobs: "force_generic" (1 = always use the generic kernels instead of the aligned
 * fast paths), "max_workspace_bytes", "host_sub_batch_bytes" (bytes staged per sub-batch of the
 * *_batch_host calls), "host_lanes" (1..4 sub-batches coded concurrently by those calls), "item_lists" (default 1:
 * the packer reads the item lists stored by the histogram pass; 0: it rebuilds them from the planes -- same bytes),
 * "huff_warp_teams" (entropy coder of framed chunks: 1 = a warp per segment when the batch has enough segments to
 * fill the GPU, default; 2 = a warp per segment whenever the segments have no parts; 0 = a CTA per segment --
 * same bytes). */
int himgcu_set_option(himgcu_ctx *ctx, const char *name, long long value);

#ifdef __cplusplus
}
#endif
#endif /* HIMG_CUDA_H_ */
