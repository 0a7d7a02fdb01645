/*
 * b200dct.h -- C ABI of the B200-native 8x8 block-transform path.
 *
 * This is the drop-in boundary for the reference's host entry points.  The reference
 * (GerryDps/CUDA-DCT-IDCT) has no FFI or header: each program forward-declares two free
 * C++ functions and calls them from main() (main_newAppr.cu:23-24,99,120).  The entry
 * points below are what a binding for that path binds; the C++ wrappers with the
 * reference's exact (mangled) signatures live in b200dct_compat.h and are implemented on
 * top of this ABI.
 *
 *   reference interface                                   replaced by
 *   ----------------------------------------------------  -------------------------------
 *   dct_all_blocks_cuda   main_newAppr.cu:252-291          b200dct_forward
 *                         main_fastAppr.cu:303-359
 *   idct_all_blocks_cuda  main_newAppr.cu:293-332          b200dct_inverse
 *                         main_fastAppr.cu:361-417
 *   dct_all_blocks        main_cublass.cu:197-260          b200dct_forward   (dense T)
 *                         main_cublass_2.cu:197-252
 *   idct_all_blocks       main_cublass.cu:265-327          b200dct_inverse   (dense T)
 *                         main_cublass_2.cu:257-311
 *   dct_* followed by idct_* (main_newAppr.cu:99,120)      b200dct_roundtrip (one fused pass)
 *   cudaMemcpyToSymbol(const_quant_matrix, ...)            b200dct_plan_set_quant
 *                         main_newAppr.cu:19,70
 *   transform_matrix device argument main_newAppr.cu:73-95 b200dct_plan_set_transform
 *   convertToFloat / convertToUnsignedChar utils.cu:10-24  dtype B200DCT_U8 on either side
 *   cudaMalloc/cudaMemcpy around the calls, main_newAppr.cu:88-95,103,124
 *                                                          b200dct_roundtrip_host
 *   the same two calls on a colour image (RGB, utils.cu:62-64)
 *     dct_all_blocks_cuda per Y/Cb/Cr plane                b200dct_forward_rgb  (RGB -> 3 zig-zag streams)
 *     idct_all_blocks_cuda per Y/Cb/Cr plane               b200dct_inverse_rgb  (3 zig-zag streams -> RGB)
 *     both, one fused pass                                 b200dct_roundtrip_rgb
 *     with 4:2:0 chroma (Cb, Cr at half resolution)        b200dct_forward_rgb420 / b200dct_inverse_rgb420
 *
 * Conventions: images are single-channel, row-major; H and W are multiples of 8 (the
 * reference silently computes garbage otherwise, main_newAppr.cu:261-262; here it is an
 * error).  Pitches are in BYTES.  All image/coefficient pointers of the device entry
 * points are caller-owned DEVICE pointers; nothing is allocated per call.  `stream` is a
 * cudaStream_t passed as void* (NULL = the legacy default stream).  Calls are
 * asynchronous on `stream` and re-entrant.  Every function returns 0 on success or a
 * negative B200DCT_ERR_* / positive cudaError_t value; nothing ever calls exit().
 * A batch of B images of H rows stored back to back is one image of B*H rows (blocks
 * are independent), so there is no batch argument.
 *
 * There is NO CPU fallback: without a CUDA device every compute entry point fails.
 */
#ifndef B200DCT_H
#define B200DCT_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200DCT_VERSION 103 /* 101: b200dct_forward_rgb / b200dct_inverse_rgb; 102: b200dct_zigzag_coded_bits flags
                               * out-of-range symbols (B200DCT_CODED_OUT_OF_RANGE), f32 metrics in 128-bit fixed point;
                               * 103: b200dct_forward_rgb420 / b200dct_inverse_rgb420 */

typedef enum b200dct_dtype {
    B200DCT_F32 = 0, /* float pixels / integer-valued float coefficients (the reference's type) */
    B200DCT_U8 = 1,  /* 8-bit pixels: convertToFloat on load, clamp+truncate on store (utils.cu:10-24) */
    /* compact coefficients; coefficient planes only.  Written values saturate to [-32768, 32767] (round to
     * nearest, then clamp).  A fused round trip's pixels come from the unsaturated coefficients: they do not
     * depend on the dtype of its coefficient output. */
    B200DCT_I16 = 2,
    /* Compact coefficient STREAM (SURVEY.md section 8f.1; the natural input of an entropy coder):
     * block-major -- block (r, c) of the H/8 x W/8 grid is 64 consecutive int16 (saturating) in
     * JPEG zig-zag scan order (ITU-T T.81 figure 5) at byte offset r*pitch + c*128.  `pitch` is
     * the bytes per BLOCK-ROW of the stream (>= (W/8)*128, multiple of 16).  Coefficient role
     * only (forward output, inverse input, round-trip coefficient output); direct kernel family. */
    B200DCT_I16_ZIGZAG = 3
} b200dct_dtype;

enum {
    B200DCT_OK = 0,
    B200DCT_ERR_ARG = -1,     /* NULL pointer, bad dtype for that role, bad plan */
    B200DCT_ERR_SHAPE = -2,   /* H or W not a positive multiple of 8, or pitch < row bytes */
    B200DCT_ERR_ALIGN = -3,   /* pointer or pitch not aligned for vector access (16 B f32/i16, 8 B u8) */
    B200DCT_ERR_NODEVICE = -4,/* no usable CUDA device */
    B200DCT_ERR_QUANT = -5,   /* Q entry not finite or zero */
    B200DCT_ERR_NOMEM = -6
};

/* Which kernel family a call may use.  AUTO picks TMA when the layout allows it
 * (f32: W % 32 == 0; u8: W % 16 == 0 ...), otherwise DIRECT. */
typedef enum b200dct_path {
    B200DCT_PATH_AUTO = 0,
    B200DCT_PATH_DIRECT = 1, /* one thread per block, vector LDG/STG */
    B200DCT_PATH_TMA = 2     /* per-warp TMA tiles through swizzled shared memory */
} b200dct_path;

/* How the INVERSE transform is evaluated when Haweel's T is in use.
 *   EXACT    : the reference's ordered FMA chains (cuda_matrix_idct, main_newAppr.cu:236-239,246-248):
 *              f32 pixels bit-identical to the reference kernels, u8 pixels bit-identical to
 *              convertToUnsignedChar (utils.cu:21) of them.
 *   FACTORED : even/odd butterfly factorisation of T^T (21 operations per 8-point transform instead
 *              of 44 FMAs).  Same mathematics, sums re-associated: the float value differs from the
 *              chain in its last bits, so an 8-bit pixel differs from the reference's by at most
 *              1 LSB, and only where the value lies within ~1e-4 of an integer (measured fraction:
 *              tests/test_gpu_factored.py, DESIGN.md section 3).  Applies to 8-bit pixel OUTPUT only;
 *              f32 pixel output always uses the chains.  The forward transform and the quantiser
 *              are never factored: quantised coefficients are bit-exact in every mode.
 *   AUTO     : FACTORED where it applies (8-bit output: the contract there is +-1 LSB), else EXACT.
 * Default AUTO. */
typedef enum b200dct_inverse_mode {
    B200DCT_INVERSE_AUTO = 0,
    B200DCT_INVERSE_EXACT = 1,
    B200DCT_INVERSE_FACTORED = 2
} b200dct_inverse_mode;

/* How a DENSE T (anything that is not bit-identical to Haweel's matrix: the "exact DCT" of the
 * cublasDCT / cublasDCTv2 variants, main_cublass.cu:85-93) is evaluated.
 *   CHAIN     : every inner product as the ascending chain of 8 FMAs (the order of the reference's
 *               non-cuBLAS kernels; bit-identical to the CPU restatement of that order with that T).
 *   SYMMETRIC : if T's even rows are symmetric and its odd rows antisymmetric (T[k][n] == +-T[k][7-n],
 *               true of the DCT-II), evaluate it through its even/odd halves: 40 instead of 64
 *               operations per 8-point transform in both directions.  Sums are re-associated; the
 *               reference for dense T is cuBLAS, whose own accumulation order is undocumented and
 *               already differs from any fixed chain in 1e-4..1e-3 of the quantised coefficients, so
 *               the criterion is the mismatch COUNT against live cuBLAS (tests/test_gpu_reference.py),
 *               pixels within 1 LSB.  A T without the structure runs CHAIN.
 *   AUTO      : SYMMETRIC where T has the structure.  Default.
 *   MMA       : the tensor-core arm (BASELINE configs[3] "CUDA-core vs tensor-core path"): f32 fused
 *               round trips run as batched 8x8 contractions on mma.sync m16n8k8 TF32 with the 2-term
 *               hi/lo split of both operands (FP32-grade inner products, FP32 accumulation); every
 *               other call of the plan runs SYMMETRIC / CHAIN.  Opt-in only: measured against the
 *               CUDA-core kernels with ncu it does not win (DESIGN.md section 6b), so AUTO never picks it. */
typedef enum b200dct_dense_mode {
    B200DCT_DENSE_AUTO = 0,
    B200DCT_DENSE_CHAIN = 1,
    B200DCT_DENSE_SYMMETRIC = 2,
    B200DCT_DENSE_MMA = 3
} b200dct_dense_mode;

typedef struct b200dct_plan b200dct_plan;

/* A plan owns the small state the reference keeps in globals: T (64 floats), Q (64
 * floats), and the retained-coefficient mask.  Defaults: Haweel's T
 * (main_newAppr.cu:73-81), the JPEG luminance Q (main_newAppr.cu:60-68), all 64
 * coefficients kept.  Plans are immutable while a call using them is being issued;
 * they hold no device memory. */
int b200dct_plan_create(b200dct_plan **plan);
void b200dct_plan_destroy(b200dct_plan *plan);

/* q: 64 floats in HOST memory, row-major Q[row*8+col] (index = threadIdx.y*8+threadIdx.x
 * in utils_kernels.cu:42,55).  Replaces cudaMemcpyToSymbol(const_quant_matrix,...). */
int b200dct_plan_set_quant(b200dct_plan *plan, const float *q);
int b200dct_plan_get_quant(const b200dct_plan *plan, float *q_out);

/* t: 64 floats in HOST memory, row-major.  If it is bit-identical to Haweel's matrix the
 * sparse compile-time kernels are used, otherwise the dense ("exact DCT") kernels. */
int b200dct_plan_set_transform(b200dct_plan *plan, const float *t);
/* Same, from a DEVICE pointer (what the reference's functions are handed); does one
 * 256-byte synchronous copy. */
int b200dct_plan_set_transform_device(b200dct_plan *plan, const void *d_t);

/* Bit (row*8+col) set <=> that quantised coefficient is kept; dropped ones are +0.0f.
 * b200dct_zigzag_mask(k) keeps the first k coefficients in JPEG zig-zag order
 * (README.md:63 of the reference: "retaining 6..10 coefficients"). */
int b200dct_plan_set_keep_mask(b200dct_plan *plan, uint64_t mask);
uint64_t b200dct_zigzag_mask(int k);

int b200dct_plan_set_path(b200dct_plan *plan, b200dct_path path);
int b200dct_plan_set_inverse(b200dct_plan *plan, b200dct_inverse_mode mode);
int b200dct_plan_set_dense(b200dct_plan *plan, b200dct_dense_mode mode);
/* Which arithmetic the plan's kernels use: 0 ordered chains (dense T), 1 Haweel's sparse
 * compile-time kernels, 2 symmetric dense kernels. */
int b200dct_plan_kernel_kind(const b200dct_plan *plan);
/* 1 if the plan's T is Haweel's matrix (sparse kernels), 0 if dense. */
int b200dct_plan_is_sparse(const b200dct_plan *plan);

/* Forward: coef = round((T.(img-128).T^T) / Q) [masked].  img: F32 or U8; coef: F32 or I16.
 * If shifted_or_null is non-NULL (F32, same pitch as img; may alias img) it receives
 * img-128, the side effect the reference leaves in its input (main_newAppr.cu:273). */
int b200dct_forward(const b200dct_plan *plan,
                    const void *img, b200dct_dtype img_dt, size_t img_pitch,
                    void *coef, b200dct_dtype coef_dt, size_t coef_pitch,
                    void *shifted_or_null,
                    int H, int W, void *stream);

/* Inverse: img = T^T.(coef*Q).T + 128.  coef: F32 or I16; img: F32 (not clamped, as the
 * reference) or U8 (clamp to [0,255] then truncate, utils.cu:21). */
int b200dct_inverse(const b200dct_plan *plan,
                    const void *coef, b200dct_dtype coef_dt, size_t coef_pitch,
                    void *img, b200dct_dtype img_dt, size_t img_pitch,
                    int H, int W, void *stream);

/* Fused forward+inverse in one HBM round trip (the headline path).  coef_or_null
 * optionally receives the quantised coefficients as well. */
int b200dct_roundtrip(const b200dct_plan *plan,
                      const void *img, b200dct_dtype in_dt, size_t in_pitch,
                      void *out, b200dct_dtype out_dt, size_t out_pitch,
                      void *coef_or_null, b200dct_dtype coef_dt, size_t coef_pitch,
                      int H, int W, void *stream);

/* Fused round trip of a BATCH of n separately allocated images of one shape and dtype (F32 or U8),
 * e.g. the 64 8192^2 images of BASELINE configs[4] or a queue of the README's 256^2..2048^2 images:
 * what a caller of the reference does with a loop of dct_all_blocks_cuda / idct_all_blocks_cuda
 * pairs over its images (main_newAppr.cu:99,120 / benchmark_fastAppr.cu:79,91 process one image per
 * program run; README.md:46 averages 100 such runs), in ONE launch per B200DCT_BATCH_MAX images
 * instead of 6 per image.
 * imgs / outs: HOST arrays of n device pointers (read before the call returns); every image obeys
 * the rules of b200dct_roundtrip (pitches shared by all images); outs[i] may equal imgs[i].
 * Results are those of n b200dct_roundtrip calls, bit for bit.  Legal under stream capture.
 * (Images large enough for the persistent TMA kernels -- F32 from 28 Mpixel -- are launched one by
 * one on that family instead, which is faster there; b200dct_last_launch_count() tells.) */
#define B200DCT_BATCH_MAX 64
int b200dct_roundtrip_batch(const b200dct_plan *plan, int n_images,
                            const void *const *imgs, void *const *outs,
                            b200dct_dtype dt, size_t in_pitch, size_t out_pitch,
                            int H, int W, void *stream);

/* Round trip for ANY image: H and W need not be multiples of 8 and nothing needs to be aligned
 * beyond the element size (SURVEY.md section 8f "generality"; the reference silently computes
 * garbage there, main_newAppr.cu:261-262).  Aligned multiples of 8 go straight to
 * b200dct_roundtrip; anything else runs ONE pass of an edge-aware kernel: blocks that stick out
 * over the right / bottom edge are completed by edge replication (what np.pad(mode="edge") gives)
 * and only their inside part is stored -- no scratch image, no extra traffic, never a wrong
 * answer.  img/out: DEVICE pointers, F32 or U8 (same dtype); out may alias img. */
int b200dct_roundtrip_any(const b200dct_plan *plan, const void *img, b200dct_dtype dt, size_t in_pitch,
                          void *out, size_t out_pitch, int H, int W, void *stream);

/* Fused round trip + quality metrics in the same pass (SURVEY.md section 8f): besides the
 * pixels (and optional coefficients) the kernel accumulates, between the pixels it read and
 * the pixels it wrote (as stored: u8 after clamp+truncate, f32 unclamped),
 *   d_acc3[0] += sum (x - y)^2     d_acc3[1] += sum x^2     d_acc3[2] += non-zero quantised coefficients
 * so MSE = acc[0]/(H*W), PEEN% = 100*sqrt(acc[0]/acc[1]) (the definitions recovered from
 * README.md:67-68 of the reference) and the coefficient density need no second pass over the
 * images.  `workspace`: device, >= b200dct_metrics_workspace_bytes, caller-owned, 8-byte aligned.  It holds
 * the call's counters when no scheduler slot is free (under stream capture with the capture pool used up,
 * or when the slot pool could not be allocated), so one workspace must not serve two calls that are in
 * flight at once.
 * `out` must not alias `img`.  Large f32 images of Haweel's T run the TMA family's metrics kernel (the
 * error is taken from the input tile in shared memory); everything else the direct family's.  Every call
 * is one launch, and its result is the same bit for bit on every path, including capture with an empty pool.
 * Range and accuracy:
 *   u8 images: exact integers.
 *   f32 images: each 8x8 block's two sums are taken in f32 in a fixed order, converted exactly to 128-bit
 *     fixed point in units of 2^-50 and added as integers, so the result does not depend on scheduling:
 *     run to run and between the two kernel families it is the same bit for bit.  The sums are exact
 *     to within 2^-50 per block, and the totals may reach 2^78 (2^22 blocks, a 16384^2 image, of pixels
 *     up to 2^20 sum to 2^68).  The relative error is that of the per-block f32 sums (measured <= 1e-6 for
 *     pixels of magnitude 2^-10 .. 2^20 with the quantiser scaled alike, tests/test_gpu_range.py). */
size_t b200dct_metrics_workspace_bytes(int H, int W);
int b200dct_roundtrip_metrics(const b200dct_plan *plan,
                              const void *img, b200dct_dtype in_dt, size_t in_pitch,
                              void *out, b200dct_dtype out_dt, size_t out_pitch,
                              void *coef_or_null, b200dct_dtype coef_dt, size_t coef_pitch,
                              int H, int W, double *d_acc3,
                              void *workspace, size_t workspace_bytes, void *stream);

/* Colour images (SURVEY.md section 8f: multi-channel / YCbCr with the chroma Q table).  The
 * reference's loader returns interleaved RGB for colour files (utils.cu:62-64: channels = 3) and
 * its programs then ignore the channel count (main_newAppr.cu:47).  This is the colour version of
 * the same fused pipeline, ONE pass over the image:
 *   RGB -> YCbCr exactly as libjpeg (the reference's image library; jccolor.c: 16-bit fixed point,
 *   8-bit samples, no subsampling), then per plane the reference's u8 pipeline (convertToFloat ->
 *   dct -> quantise -> dequantise -> idct -> convertToUnsignedChar) with the plan's luminance table
 *   for Y and its chrominance table (default ITU-T T.81 Annex K.2) for Cb and Cr, then YCbCr -> RGB
 *   exactly as libjpeg's decoder (jdcolor.c).
 * rgb/out: DEVICE pointers, H x W pixels of 3 bytes, 8-byte aligned rows (pitch in bytes, % 8 == 0).
 * zz3_or_null: optionally the three block-major zig-zag int16 coefficient streams (Y, Cb, Cr;
 * layout of B200DCT_I16_ZIGZAG), zz_plane_bytes apart (>= H*W*2, % 16 == 0).  The plan's mask
 * applies to all three planes; its inverse mode as for 8-bit grey images (EXACT: planes
 * bit-identical to the reference's arithmetic).  Haweel's T only (B200DCT_ERR_ARG otherwise). */
int b200dct_plan_set_chroma_quant(b200dct_plan *plan, const float q[64]);
int b200dct_plan_get_chroma_quant(const b200dct_plan *plan, float q[64]);
int b200dct_roundtrip_rgb(const b200dct_plan *plan, const void *rgb, size_t in_pitch,
                          void *out, size_t out_pitch, void *zz3_or_null, size_t zz_plane_bytes,
                          int H, int W, void *stream);
/* The two halves of b200dct_roundtrip_rgb, split at the coefficient streams, for callers that store
 * or send the compact coefficients, size them (b200dct_zigzag_coded_bits) or change them before
 * decoding -- what the reference's caller can do between its two calls (main_newAppr.cu:103).
 * Arguments, stream layout and error codes as b200dct_roundtrip_rgb; zz3 is required.  One launch
 * each (b200dct_last_path() "rgb"), legal under stream capture.  b200dct_inverse_rgb of the streams
 * b200dct_forward_rgb wrote gives b200dct_roundtrip_rgb's pixels bit for bit, in either inverse mode,
 * as long as no stream value saturates (never for Q entries >= 1/16).  Beyond that the streams hold the
 * saturated values while b200dct_roundtrip_rgb's pixels still come from the unsaturated ones.
 * RGB -> YCbCr (libjpeg jccolor.c) -> per plane convertToFloat, dct, quantise (luminance Q for Y,
 * chrominance Q for Cb/Cr, plan's keep mask) -> three block-major zig-zag int16 streams
 * (B200DCT_I16_ZIGZAG layout, block-row pitch (W/8)*128, planes zz_plane_bytes apart). */
int b200dct_forward_rgb(const b200dct_plan *plan, const void *rgb, size_t in_pitch,
                        void *zz3, size_t zz_plane_bytes, int H, int W, void *stream);
/* three zig-zag streams -> per plane dequantise, idct, convertToUnsignedChar (plan's inverse mode)
 * -> YCbCr -> RGB (libjpeg jdcolor.c). */
int b200dct_inverse_rgb(const b200dct_plan *plan, const void *zz3, size_t zz_plane_bytes,
                        void *out, size_t out_pitch, int H, int W, void *stream);
/* 4:2:0 chroma subsampling, what libjpeg and every JPEG encoder do by default: Cb and Cr at half the
 * resolution in both directions, so a 16x16 macroblock (MCU) carries four Y blocks and one Cb and one Cr
 * block -- half the coefficients of 4:4:4.  The resampling is libjpeg's, bit for bit: the encoder's
 * h2v2_downsample (jcsample.c: a half-resolution sample is (a + b + c + d + bias) >> 2 over its 2x2 group of
 * 8-bit samples, bias 1 at even and 2 at odd output columns) and the decoder's default h2v2_fancy_upsample
 * (jdsample.c: triangle filter 3/4, 1/4 in both directions, edges replicated).
 * rgb/out: as b200dct_roundtrip_rgb (interleaved RGB u8, 8-byte aligned rows, pitch in bytes).  H and W
 * are positive multiples of 16 (B200DCT_ERR_SHAPE otherwise, and for a pitch below W*3).  Three separate
 * block-major zig-zag int16 streams (B200DCT_I16_ZIGZAG layout), tightly packed, 16-byte aligned
 * (B200DCT_ERR_ALIGN otherwise, as for misaligned pixel pointers or pitches): zz_y holds H/8 x W/8 blocks
 * with a block-row pitch of (W/8)*128 bytes, zz_cb and zz_cr H/16 x W/16 blocks with a pitch of
 * (W/16)*128 bytes.  NULL pointers and a dense T give B200DCT_ERR_ARG (Haweel's T only).  One launch
 * each (b200dct_last_path() "rgb"), legal under stream capture.
 * Forward: RGB -> YCbCr (jccolor.c) -> 2x2 downsampling of Cb and Cr -> per plane convertToFloat, dct,
 * quantise (luminance Q for Y, chrominance Q for Cb and Cr, the plan's keep mask on all three).
 * Inverse: per plane dequantise, idct (the plan's inverse mode), convertToUnsignedChar -> upsampling of Cb
 * and Cr -> YCbCr -> RGB (jdcolor.c).
 * Coded size: b200dct_zigzag_coded_bits of zz_y with table 0 (H, W), plus zz_cb and zz_cr with table 1 at
 * (H/2, W/2), is exactly the entropy-coded size of a baseline JPEG with three non-interleaved scans, one per
 * component (sampling factors 2x2, 1x1, 1x1): in such a scan a component's blocks come in raster order
 * (ITU-T T.81 A.2.2), as that function counts them. */
int b200dct_forward_rgb420(const b200dct_plan *plan, const void *rgb, size_t in_pitch,
                           void *zz_y, void *zz_cb, void *zz_cr, int H, int W, void *stream);
int b200dct_inverse_rgb420(const b200dct_plan *plan, const void *zz_y, const void *zz_cb, const void *zz_cr,
                           void *out, size_t out_pitch, int H, int W, void *stream);

/* Size in BITS of the baseline-JPEG entropy-coded scan (ITU-T T.81 sequential Huffman with the
 * Annex K.3 tables, i.e. what libjpeg writes with optimize off; no headers, stuffing or padding)
 * of one plane's zig-zag stream (B200DCT_I16_ZIGZAG layout; pitch = bytes per block-row), ADDED
 * to *d_bits (device, 8-byte aligned).  table: 0 luminance codes, 1 chrominance codes.  This
 * defines the "Compr. Factor" of the reference's README (README.md:62-69), for which the
 * reference has no code:  CF = 8 * H * W / bits.
 * Baseline JPEG codes DC differences of magnitude <= 2047 (categories 0..11) and AC values of
 * magnitude <= 1023 (categories 1..10) only.  A stream with any other symbol -- which quantiser
 * entries below 1 can produce from 8-bit pixels -- has no baseline size: its symbols count 0 bits
 * and the call ORs B200DCT_CODED_OUT_OF_RANGE (bit 63) into *d_bits. */
#define B200DCT_CODED_OUT_OF_RANGE (1ull << 63)
int b200dct_zigzag_coded_bits(const void *zz, size_t pitch, int H, int W, int table,
                              unsigned long long *d_bits, void *stream);

/* Host-buffer round trip: what the reference's main() does around its two calls
 * (cudaMalloc, H2D, dct, idct, D2H: main_newAppr.cu:88-124), as one call on the current
 * device.  h_in/h_out are HOST pointers (pinned or pageable), tightly packed rows.
 * Internally the image is cut into block-row chunks that are copied, transformed and
 * copied back on rotating streams so H2D, kernel and D2H overlap.  Synchronous.  The calling
 * thread keeps one pipeline (4 streams, 8 chunk buffers) per device until it exits or calls
 * b200dct_host_release(). */
int b200dct_roundtrip_host(const b200dct_plan *plan,
                           const void *h_in, b200dct_dtype in_dt,
                           void *h_out, b200dct_dtype out_dt,
                           int H, int W);
int b200dct_host_release(void);
int b200dct_host_last_launch_count(void); /* kernels launched by this thread's last b200dct_roundtrip_host */

/* The same pipeline as an object, for callers that process a SEQUENCE of images (the reference
 * programs handle one image per process, main_newAppr.cu:26-165; a service handles many):
 * b200dct_host_pipeline_submit only enqueues the image's chunks and returns, so consecutive images
 * overlap -- image i+1 is uploading while image i is still coming back -- and the per-image
 * fill/drain bubble of the synchronous call disappears.  h_in must stay valid and h_out must not
 * be read until b200dct_host_pipeline_wait(ticket) (or _drain) returns; pinned host memory is
 * needed for the copies to be asynchronous (pageable memory works, submit then blocks).
 * A pipeline belongs to the device that was current at creation and to one submitting thread at a
 * time.  chunk_bytes = 0: default (64 MiB, env B200DCT_PIPE_CHUNK_MB); slots = 0: default (3);
 * device memory held: 2 * slots * chunk_bytes.
 * A chunk must hold at least one block-row (8 * W * element size), else B200DCT_ERR_SHAPE. */
typedef struct b200dct_host_pipeline b200dct_host_pipeline;
int  b200dct_host_pipeline_create(b200dct_host_pipeline **out, size_t chunk_bytes, int slots);
void b200dct_host_pipeline_destroy(b200dct_host_pipeline *pipe);   /* waits for what is in flight */
size_t b200dct_host_pipeline_chunk_bytes(const b200dct_host_pipeline *pipe);
int  b200dct_host_pipeline_submit(b200dct_host_pipeline *pipe, const b200dct_plan *plan,
                                  const void *h_in, b200dct_dtype in_dt,
                                  void *h_out, b200dct_dtype out_dt,
                                  int H, int W, unsigned long long *ticket_or_null);
int  b200dct_host_pipeline_wait(b200dct_host_pipeline *pipe, unsigned long long ticket);
int  b200dct_host_pipeline_drain(b200dct_host_pipeline *pipe);
int  b200dct_host_pipeline_last_launch_count(const b200dct_host_pipeline *pipe);

/* Sum of squared error and signal energy between two device images (same dtype,
 * F32 or U8), accumulated in double: MSE = sse/N, PEEN% = 100*sqrt(sse/energy)
 * (the definitions recovered from README.md:67-68 of the reference).
 * d_acc: device pointer to 2 doubles {sse, energy}; the call ADDS into it. */
int b200dct_metrics_accumulate(const void *ref_img, const void *test_img, b200dct_dtype dt,
                               size_t pitch, int H, int W, double *d_acc, void *stream);

/* Measurement helper: average device milliseconds of `iters` back-to-back identical calls
 * (CUDA events on `stream`, launched from C so no interpreter sits between launches).
 * which: 0 roundtrip(a -> b, optional coefficient plane c), 1 forward(a -> b),
 * 2 inverse(a -> b), 3 forward(a -> c) followed by inverse(c -> b) (the reference's
 * two-call sequence, main_newAppr.cu:99,120). */
int b200dct_time_calls(const b200dct_plan *plan, int which,
                       const void *a, b200dct_dtype a_dt, size_t a_pitch,
                       void *b, b200dct_dtype b_dt, size_t b_pitch,
                       void *c, b200dct_dtype c_dt, size_t c_pitch,
                       int H, int W, int iters, float *ms_per_iter, void *stream);

/* Self-test of the kernels' constant-divisor division: sweeps the float bit patterns
 * [first, first+count) as dividends against __fdiv_rn (the reference's div.rn.f32,
 * utils_kernels.cu:42) for divisor d.  ADDS into d_out2 (device, 2 x uint64):
 * [0] quotients whose bits differ for |x| >= 2^-120, [1] quantised values roundf(q) that
 * differ (x = -0.0f, which the transform cannot produce, is skipped). */
int b200dct_selftest_division(float d, unsigned long long first, unsigned long long count,
                              unsigned long long *d_out2, void *stream);

/* How many kernels the last call on this thread launched (for bench accounting). */
int b200dct_last_launch_count(void);
/* Kernels launched under stream capture by the persistent (TMA) family own a scheduler slot for the
 * life of the process (4096 per device; a graph replays its slot, CUDA has no destroy hook to hand
 * it back).  Returns how many are left on the current device; at 0 captured AUTO launches run the
 * direct kernel family instead (about 5 % slower at 8192^2), b200dct_last_path() reports which. */
int b200dct_capture_slots_left(void);
/* Name of the kernel family the last call on this thread used: "tma", "direct" or "any". */
const char *b200dct_last_path(void);

const char *b200dct_error_string(int err);
int b200dct_version(void);

#ifdef __cplusplus
}
#endif
#endif /* B200DCT_H */
