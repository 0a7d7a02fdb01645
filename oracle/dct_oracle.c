/*
 * dct_oracle.c -- CPU restatement of the reference's 8x8 block-transform path.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing in the product path (the package, the C-ABI
 * library, the compat wrappers) may import, link or execute this file.  It is used
 * by tests/, by __graft_entry__.smoke() and by bench.py's cpu_baseline / reference
 * legs as the *checker* and as the sequential CPU baseline.
 *
 * Parity status: the reference ships NO tests, golden vectors or fixtures
 * (SURVEY.md section 4).  This restatement is pinned instead by running the
 * reference's own kernels, compiled unmodified from /root/reference into
 * oracle/_ref/ (see oracle/Makefile), on a B200 and comparing bit-for-bit
 * (tests/test_gpu_reference.py), and by the committed fixtures in tests/golden/.
 *
 * Each function cites the reference file:line it follows.  Arithmetic contract
 * (SURVEY.md Appendix A): all values are IEEE binary32; every inner product is an
 * ordered chain of 8 fused multiply-adds starting from +0.0f with the summation
 * index ascending (that is what nvcc emits for the reference's `sums += a*b` loops
 * under its default -fmad=true); quantisation is a correctly-rounded division
 * followed by round-half-away-from-zero; dequantisation is a plain multiply.
 *
 * Build: gcc -O2 -ffp-contract=off (so that ONLY the explicit fmaf() calls fuse).
 * The hot loops are cloned for FMA-capable CPUs via target_clones, the default
 * clone falls back to glibc's correctly-rounded software fmaf().
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define BS 8

#if defined(__x86_64__) && defined(__GNUC__)
#define ORACLE_CLONES __attribute__((target_clones("fma", "default")))
#else
#define ORACLE_CLONES
#endif

/* Haweel's approximate-DCT matrix exactly as the reference spells it
 * (main_newAppr.cu:73-81): double literals narrowed to float. */
static const float k_haweel_T[64] = {
    0.35355339, 0.35355339, 0.35355339, 0.35355339, 0.35355339, 0.35355339, 0.35355339, 0.35355339,
    0.5, 0.5, 0, 0, 0, 0, -0.5, -0.5,
    0.4472136, 0.2236068, -0.2236068, -0.4472136, -0.4472136, -0.2236068, 0.2236068, 0.4472136,
    0, 0, -0.70710678, 0, 0, 0.70710678, 0, 0,
    0.35355339, -0.35355339, -0.35355339, 0.35355339, 0.35355339, -0.35355339, -0.35355339, 0.35355339,
    0.5, -0.5, 0, 0, 0, 0, 0.5, -0.5,
    0.2236068, -0.4472136, 0.4472136, -0.2236068, -0.2236068, 0.4472136, -0.4472136, 0.2236068,
    0, 0, 0, -0.70710678, 0.70710678, 0, 0, 0};

/* JPEG luminance quantisation table (main_newAppr.cu:60-68). */
static const float k_jpeg_Q[64] = {
    16, 11, 10, 16, 24, 40, 51, 61,
    12, 12, 14, 19, 26, 58, 60, 55,
    14, 13, 16, 24, 40, 57, 69, 56,
    14, 17, 22, 29, 51, 87, 80, 62,
    18, 22, 37, 56, 68, 109, 103, 77,
    24, 35, 55, 64, 81, 104, 113, 92,
    49, 64, 78, 87, 103, 121, 120, 101,
    72, 92, 95, 98, 112, 100, 103, 99};

/* JPEG zig-zag scan order as (row*8+col); the retained-coefficient mask keeps the
 * first k entries (SURVEY.md section 8c; README.md:63 of the reference). */
static const unsigned char k_zigzag[64] = {
    0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5,
    12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21, 28,
    35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51,
    58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};

const float *oracle_haweel_T(void) { return k_haweel_T; }
const float *oracle_jpeg_Q(void) { return k_jpeg_Q; }

/* True orthonormal DCT-II matrix in float ("exact DCT" = the dense variants fed a
 * real DCT matrix, SURVEY.md S3).  Computed in double, narrowed once. */
void oracle_dct2_T(float *T)
{
    for (int k = 0; k < BS; k++)
        for (int n = 0; n < BS; n++) {
            double c = (k == 0) ? sqrt(1.0 / BS) : sqrt(2.0 / BS);
            T[k * BS + n] = (float)(c * cos((2 * n + 1) * k * M_PI / (2.0 * BS)));
        }
}

/* Bit i of the mask <=> coefficient at (row*8+col)==i is kept. */
uint64_t oracle_zigzag_mask(int k)
{
    uint64_t m = 0;
    if (k >= 64) return ~(uint64_t)0;
    for (int i = 0; i < k; i++) m |= (uint64_t)1 << k_zigzag[i];
    return m;
}

/* Compact coefficient stream (SURVEY.md section 8f.1; not in the reference, whose coefficient
 * plane is a float image, main_newAppr.cu:99-103): block-major, block (r,c) -> 64 consecutive
 * int16 in zig-zag order, values = the integer-valued float coefficients saturated to int16. */
void oracle_zigzag_i16(const float *coef, int H, int W, int16_t *out)
{
    const int bx = W / BS;
    for (int r = 0; r < H / BS; r++)
        for (int c = 0; c < bx; c++)
            for (int k = 0; k < 64; k++) {
                float v = coef[(size_t)(r * BS + k_zigzag[k] / BS) * W + c * BS + k_zigzag[k] % BS];
                if (v > 32767.0f) v = 32767.0f;
                if (v < -32768.0f) v = -32768.0f;
                out[((size_t)r * bx + c) * 64 + k] = (int16_t)lrintf(v);
            }
}
/* and back: the float coefficient plane the inverse transform starts from */
void oracle_unzigzag_i16(const int16_t *in, int H, int W, float *coef)
{
    const int bx = W / BS;
    for (int r = 0; r < H / BS; r++)
        for (int c = 0; c < bx; c++)
            for (int k = 0; k < 64; k++)
                coef[(size_t)(r * BS + k_zigzag[k] / BS) * W + c * BS + k_zigzag[k] % BS] =
                    (float)in[((size_t)r * bx + c) * 64 + k];
}

/* Reference input generator: srand(seed); img[i*N+j] = rand()%256
 * (Benchmark_code/benchmark_fastAppr.cu:44-47).  glibc rand(). */
void oracle_fill_rand(float *img, size_t n, unsigned seed)
{
    srand(seed);
    for (size_t i = 0; i < n; i++) img[i] = (float)(rand() % 256);
}

void oracle_fill_rand_u8(unsigned char *img, size_t n, unsigned seed)
{
    srand(seed);
    for (size_t i = 0; i < n; i++) img[i] = (unsigned char)(rand() % 256);
}

/* utils.cu:10-15 */
void oracle_convert_to_float(const unsigned char *in, float *out, size_t n)
{
    for (size_t i = 0; i < n; i++) out[i] = (float)in[i];
}

/* utils.cu:18-24 : clamp to [0,255] then C cast (truncation toward zero). */
void oracle_convert_to_u8(const float *in, unsigned char *out, size_t n)
{
    for (size_t i = 0; i < n; i++) out[i] = (unsigned char)fminf(fmaxf(in[i], 0.0f), 255.0f);
}

/* ---- one block-row strip of the forward path -------------------------------------
 * sub_matrix_scalar   utils_kernels.cu:8-18     X = img - 128
 * cuda_matrix_dct     main_newAppr.cu:177-211   M = T.X (:193-197), Y = M.T^T (:206-209)
 * divide_matrices     utils_kernels.cu:34-44    C = round(Y / Q[ty*8+tx])
 * `keep` is applied to the quantised coefficients (exact +0.0f where dropped).
 */
ORACLE_CLONES
static void fwd_block(const float *src, size_t pitch, const float *T, const float *Q,
                      uint64_t keep, float *dst, size_t dpitch, float *shifted, size_t spitch)
{
    float X[BS][BS], M[BS][BS];
    for (int y = 0; y < BS; y++)
        for (int x = 0; x < BS; x++) {
            X[y][x] = src[y * pitch + x] - 128.0f;
            if (shifted) shifted[y * spitch + x] = X[y][x];
        }
    for (int y = 0; y < BS; y++)
        for (int x = 0; x < BS; x++) {
            float s = 0.0f;
            for (int i = 0; i < BS; i++) s = fmaf(T[y * BS + i], X[i][x], s);
            M[y][x] = s;
        }
    for (int y = 0; y < BS; y++)
        for (int x = 0; x < BS; x++) {
            float s = 0.0f;
            for (int i = 0; i < BS; i++) s = fmaf(M[y][i], T[x * BS + i], s);
            float c = roundf(s / Q[y * BS + x]);
            if (!((keep >> (y * BS + x)) & 1)) c = 0.0f;
            dst[y * dpitch + x] = c;
        }
}

/* ---- inverse path -----------------------------------------------------------------
 * multiply_matrices   utils_kernels.cu:47-57    D = C * Q[ty*8+tx]
 * cuda_matrix_idct    main_newAppr.cu:220-250   M = T^T.D (:236-239), R = M.T (:246-248)
 * add_matrix_scalar   utils_kernels.cu:21-31    out = R + 128   (not clamped)
 */
ORACLE_CLONES
static void inv_block(const float *src, size_t pitch, const float *T, const float *Q,
                      float *dst, size_t dpitch)
{
    float D[BS][BS], M[BS][BS];
    for (int y = 0; y < BS; y++)
        for (int x = 0; x < BS; x++) D[y][x] = src[y * pitch + x] * Q[y * BS + x];
    for (int y = 0; y < BS; y++)
        for (int x = 0; x < BS; x++) {
            float s = 0.0f;
            for (int i = 0; i < BS; i++) s = fmaf(T[i * BS + y], D[i][x], s);
            M[y][x] = s;
        }
    for (int y = 0; y < BS; y++)
        for (int x = 0; x < BS; x++) {
            float s = 0.0f;
            for (int i = 0; i < BS; i++) s = fmaf(M[y][i], T[i * BS + x], s);
            dst[y * dpitch + x] = s + 128.0f;
        }
}

/* dct_all_blocks_cuda (main_newAppr.cu:252-291).  If `shifted` is non-NULL it
 * receives img-128, the value the reference leaves in its (mutated) input buffer
 * (:273).  threads<=1 -> sequential. */
void oracle_dct(const float *img, int H, int W, const float *T, const float *Q,
                uint64_t keep, float *coef, float *shifted, int threads)
{
    const int by = H / BS, bx = W / BS;
#ifdef _OPENMP
#pragma omp parallel for schedule(static) num_threads(threads > 1 ? threads : 1)
#endif
    for (int r = 0; r < by; r++)
        for (int c = 0; c < bx; c++) {
            size_t off = (size_t)r * BS * W + (size_t)c * BS;
            fwd_block(img + off, W, T, Q, keep, coef + off, W,
                      shifted ? shifted + off : NULL, W);
        }
    (void)threads;
}

/* idct_all_blocks_cuda (main_newAppr.cu:293-332). */
void oracle_idct(const float *coef, int H, int W, const float *T, const float *Q,
                 float *out, int threads)
{
    const int by = H / BS, bx = W / BS;
#ifdef _OPENMP
#pragma omp parallel for schedule(static) num_threads(threads > 1 ? threads : 1)
#endif
    for (int r = 0; r < by; r++)
        for (int c = 0; c < bx; c++) {
            size_t off = (size_t)r * BS * W + (size_t)c * BS;
            inv_block(coef + off, W, T, Q, out + off, W);
        }
    (void)threads;
}

/* Fused round trip on float pixels: coef (optional) and reconstructed pixels. */
void oracle_roundtrip(const float *img, int H, int W, const float *T, const float *Q,
                      uint64_t keep, float *coef_or_null, float *out, int threads)
{
    const int by = H / BS, bx = W / BS;
#ifdef _OPENMP
#pragma omp parallel for schedule(static) num_threads(threads > 1 ? threads : 1)
#endif
    for (int r = 0; r < by; r++)
        for (int c = 0; c < bx; c++) {
            float tmp[BS * BS];
            size_t off = (size_t)r * BS * W + (size_t)c * BS;
            fwd_block(img + off, W, T, Q, keep, tmp, BS, NULL, 0);
            if (coef_or_null)
                for (int y = 0; y < BS; y++)
                    memcpy(coef_or_null + off + (size_t)y * W, tmp + y * BS, BS * sizeof(float));
            inv_block(tmp, BS, T, Q, out + off, W);
        }
    (void)threads;
}

/* u8 in -> u8 out round trip: convertToFloat, forward, inverse, convertToUnsignedChar
 * (main_newAppr.cu:47,99,120,141). */
void oracle_roundtrip_u8(const unsigned char *img, int H, int W, const float *T,
                         const float *Q, uint64_t keep, float *coef_or_null,
                         unsigned char *out, int threads)
{
    const int by = H / BS, bx = W / BS;
#ifdef _OPENMP
#pragma omp parallel for schedule(static) num_threads(threads > 1 ? threads : 1)
#endif
    for (int r = 0; r < by; r++)
        for (int c = 0; c < bx; c++) {
            float blk[BS * BS], tmp[BS * BS], rec[BS * BS];
            size_t off = (size_t)r * BS * W + (size_t)c * BS;
            for (int y = 0; y < BS; y++)
                oracle_convert_to_float(img + off + (size_t)y * W, blk + y * BS, BS);
            fwd_block(blk, BS, T, Q, keep, tmp, BS, NULL, 0);
            if (coef_or_null)
                for (int y = 0; y < BS; y++)
                    memcpy(coef_or_null + off + (size_t)y * W, tmp + y * BS, BS * sizeof(float));
            inv_block(tmp, BS, T, Q, rec, BS);
            for (int y = 0; y < BS; y++)
                oracle_convert_to_u8(rec + y * BS, out + off + (size_t)y * W, BS);
        }
    (void)threads;
}

/* ---- colour images (SURVEY.md section 8f "generality": multi-channel / YCbCr with the chroma
 * table) --------------------------------------------------------------------------------------
 * The reference's loader hands back interleaved RGB for colour files (utils.cu:62-64:
 * `*channels = cinfo.output_components; // 1 for grayscale, 3 for RGB`) and its programs then
 * ignore the channel count (main_newAppr.cu:47).  The path below is what a JPEG-style codec does
 * with such a buffer, built only from pieces the reference already contains or links:
 *   1. RGB -> YCbCr exactly as libjpeg does it (the reference's image dependency, jpeglib.h,
 *      utils.cu:6; IJG libjpeg / libjpeg-turbo jccolor.c rgb_ycc_convert: 16-bit fixed point,
 *      SCALEBITS = 16, FIX(x) = (int)(x * 65536 + 0.5), ONE_HALF rounding; Cb/Cr add
 *      CBCR_OFFSET + ONE_HALF - 1), samples are u8, no subsampling (4:4:4);
 *   2. every plane goes through the reference's own u8 pipeline (convertToFloat utils.cu:10-15,
 *      dct_all_blocks_cuda, idct_all_blocks_cuda, convertToUnsignedChar utils.cu:18-24) with the
 *      luminance table for Y (main_newAppr.cu:60-68) and the ITU-T T.81 Annex K.2 chrominance
 *      table for Cb and Cr;
 *   3. YCbCr -> RGB exactly as libjpeg's decoder (jdcolor.c ycc_rgb_convert / build_ycc_rgb_table).
 * Pinned: steps 1 and 3 against the real libjpeg (libjpeg-turbo inside Pillow) through
 * tests/golden/libjpeg_color.npz (tests/golden/make_libjpeg_color_golden.py), zero mismatches;
 * step 2 is the pinned grayscale path. */
static const float k_jpeg_Q_chroma[64] = {
    17, 18, 24, 47, 99, 99, 99, 99,
    18, 21, 26, 66, 99, 99, 99, 99,
    24, 26, 56, 99, 99, 99, 99, 99,
    47, 66, 99, 99, 99, 99, 99, 99,
    99, 99, 99, 99, 99, 99, 99, 99,
    99, 99, 99, 99, 99, 99, 99, 99,
    99, 99, 99, 99, 99, 99, 99, 99,
    99, 99, 99, 99, 99, 99, 99, 99};
const float *oracle_jpeg_Q_chroma(void) { return k_jpeg_Q_chroma; }

#define CFIX(x) ((int32_t)((x) * 65536.0 + 0.5))
/* jccolor.c: rgb_ycc_start tables folded into one expression per sample */
void oracle_rgb_to_ycc(const unsigned char *rgb, size_t npix, unsigned char *y, unsigned char *cb, unsigned char *cr)
{
    for (size_t i = 0; i < npix; i++) {
        const int32_t r = rgb[3 * i], g = rgb[3 * i + 1], b = rgb[3 * i + 2];
        y[i] = (unsigned char)((CFIX(0.29900) * r + CFIX(0.58700) * g + CFIX(0.11400) * b + 32768) >> 16);
        cb[i] = (unsigned char)((-CFIX(0.16874) * r - CFIX(0.33126) * g + CFIX(0.50000) * b + (128 << 16) + 32767) >> 16);
        cr[i] = (unsigned char)((CFIX(0.50000) * r - CFIX(0.41869) * g - CFIX(0.08131) * b + (128 << 16) + 32767) >> 16);
    }
}
static unsigned char clamp_u8(int32_t v) { return (unsigned char)(v < 0 ? 0 : (v > 255 ? 255 : v)); }
/* jdcolor.c: Cr_r_tab, Cb_b_tab are rounded and shifted per table entry, the two green terms
 * share one shift (Cb_g_tab carries the ONE_HALF); >> on negative values is arithmetic */
void oracle_ycc_to_rgb(const unsigned char *y, const unsigned char *cb, const unsigned char *cr, size_t npix, unsigned char *rgb)
{
    for (size_t i = 0; i < npix; i++) {
        const int32_t yy = y[i], b = (int32_t)cb[i] - 128, r = (int32_t)cr[i] - 128;
        rgb[3 * i] = clamp_u8(yy + ((CFIX(1.40200) * r + 32768) >> 16));
        rgb[3 * i + 1] = clamp_u8(yy + ((-CFIX(0.34414) * b + 32768 - CFIX(0.71414) * r) >> 16));
        rgb[3 * i + 2] = clamp_u8(yy + ((CFIX(1.77200) * b + 32768) >> 16));
    }
}

void oracle_roundtrip_u8(const unsigned char *img, int H, int W, const float *T, const float *Q, uint64_t keep,
                         float *coef_or_null, unsigned char *out, int threads);

/* Interleaved RGB u8 in -> interleaved RGB u8 out.  planes_or_null: 3*H*W bytes, the Y, Cb, Cr
 * planes AFTER the round trip (what step 3 consumes); coef3_or_null: 3*H*W floats, the quantised
 * coefficient planes of Y, Cb, Cr. */
void oracle_roundtrip_rgb(const unsigned char *rgb, int H, int W, const float *T, const float *Qluma,
                          const float *Qchroma, uint64_t keep, unsigned char *out, unsigned char *planes_or_null,
                          float *coef3_or_null, int threads)
{
    const size_t n = (size_t)H * W;
    unsigned char *in3 = (unsigned char *)malloc(3 * n), *out3 = planes_or_null ? planes_or_null : (unsigned char *)malloc(3 * n);
    oracle_rgb_to_ycc(rgb, n, in3, in3 + n, in3 + 2 * n);
    for (int c = 0; c < 3; c++)
        oracle_roundtrip_u8(in3 + c * n, H, W, T, c == 0 ? Qluma : Qchroma, keep, coef3_or_null ? coef3_or_null + c * n : NULL,
                            out3 + c * n, threads);
    oracle_ycc_to_rgb(out3, out3 + n, out3 + 2 * n, n, out);
    free(in3);
    if (!planes_or_null) free(out3);
}

/* ---- compression factor -------------------------------------------------------------------
 * The reference's README reports a "Compr. Factor" per retained-coefficient setting
 * (README.md:62-69) without code for it.  Definition used here (SURVEY.md section 8f.1: the compact
 * coefficient stream "gives the README's compression factor a definition"):
 *     CF = 8 * H * W / (size in bits of the baseline-JPEG entropy-coded scan of the coefficients)
 * i.e. ITU-T T.81 sequential Huffman coding with the Annex K.3 "typical" tables -- the tables
 * libjpeg writes (jstdhuff.c; pinned through tests/golden/libjpeg_color.npz, extracted from a
 * file written by the real libjpeg): per block the DC difference to the previous block of the
 * plane in raster order (category code + category bits), then the AC coefficients in zig-zag
 * order as (run, size) codes + size bits, ZRL (0xF0) for every 16 zeros in front of a non-zero
 * coefficient, EOB (0x00) when the block ends in zeros.  Byte stuffing, padding and headers are
 * not counted.  table 0 = luminance codes, 1 = chrominance codes. */
static const unsigned char k_dc_bits[2][16] = {{0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0},
                                               {0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0}};
static const unsigned char k_ac_bits[2][16] = {{0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 0x7d},
                                               {0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 0x77}};
static const unsigned char k_ac_vals[2][162] = {
    {0x01, 0x02, 0x03, 0x00, 0x04, 0x11, 0x05, 0x12, 0x21, 0x31, 0x41, 0x06, 0x13, 0x51, 0x61, 0x07, 0x22, 0x71,
     0x14, 0x32, 0x81, 0x91, 0xa1, 0x08, 0x23, 0x42, 0xb1, 0xc1, 0x15, 0x52, 0xd1, 0xf0, 0x24, 0x33, 0x62, 0x72,
     0x82, 0x09, 0x0a, 0x16, 0x17, 0x18, 0x19, 0x1a, 0x25, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x34, 0x35, 0x36, 0x37,
     0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59,
     0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a, 0x83,
     0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a, 0xa2, 0xa3,
     0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3,
     0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe1, 0xe2,
     0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf1, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa},
    {0x00, 0x01, 0x02, 0x03, 0x11, 0x04, 0x05, 0x21, 0x31, 0x06, 0x12, 0x41, 0x51, 0x07, 0x61, 0x71, 0x13, 0x22,
     0x32, 0x81, 0x08, 0x14, 0x42, 0x91, 0xa1, 0xb1, 0xc1, 0x09, 0x23, 0x33, 0x52, 0xf0, 0x15, 0x62, 0x72, 0xd1,
     0x0a, 0x16, 0x24, 0x34, 0xe1, 0x25, 0xf1, 0x17, 0x18, 0x19, 0x1a, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x35, 0x36,
     0x37, 0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58,
     0x59, 0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a,
     0x82, 0x83, 0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a,
     0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba,
     0xc2, 0xc3, 0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda,
     0xe2, 0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa}};

/* tables as the DHT marker carries them: which 0 DC / 1 AC; table 0 luminance / 1 chrominance */
void oracle_huffman_spec(int which, int table, unsigned char bits16[16], unsigned char *vals, int *nvals)
{
    memcpy(bits16, which ? k_ac_bits[table] : k_dc_bits[table], 16);
    int n = 0;
    for (int i = 0; i < 16; i++) n += bits16[i];
    for (int i = 0; i < n; i++) vals[i] = which ? k_ac_vals[table][i] : (unsigned char)i;
    *nvals = n;
}

/* code length in bits of every symbol (0 = symbol has no code): T.81 Annex C, codes of length
 * l are assigned to the next BITS[l] values in HUFFVAL order */
void oracle_huffman_lengths(int which, int table, unsigned char len256[256])
{
    unsigned char bits[16], vals[256];
    int n, k = 0;
    oracle_huffman_spec(which, table, bits, vals, &n);
    memset(len256, 0, 256);
    for (int l = 1; l <= 16; l++)
        for (int i = 0; i < bits[l - 1]; i++) len256[vals[k++]] = (unsigned char)l;
}

static int bit_size(int v) /* T.81 F.1.2.1: SSSS = number of bits of |v| */
{
    int a = v < 0 ? -v : v, n = 0;
    while (a) { n++; a >>= 1; }
    return n;
}

/* stream: the block-major zig-zag int16 stream of ONE plane (oracle_zigzag_i16), blocks in raster order.
 * Baseline JPEG codes DC-difference categories 0..11 and AC categories 1..10 only: a symbol outside them
 * has no code, counts 0 bits and sets bit 63 of the result (b200dct_zigzag_coded_bits does the same). */
uint64_t oracle_coded_bits(const int16_t *stream, size_t nblocks, int table)
{
    unsigned char dcl[256], acl[256];
    oracle_huffman_lengths(0, table, dcl);
    oracle_huffman_lengths(1, table, acl);
    uint64_t bits = 0, out_of_range = 0;
    int prev = 0;
    for (size_t b = 0; b < nblocks; b++) {
        const int16_t *c = stream + b * 64;
        const int s = bit_size((int)c[0] - prev);
        prev = c[0];
        if (s <= 11) bits += dcl[s] + s;
        else out_of_range = 1;
        int run = 0;
        for (int k = 1; k < 64; k++) {
            if (c[k] == 0) { run++; continue; }
            while (run > 15) { bits += acl[0xf0]; run -= 16; }
            const int sz = bit_size(c[k]);
            if (sz <= 10) bits += acl[(run << 4) | sz] + sz;
            else out_of_range = 1;
            run = 0;
        }
        if (run) bits += acl[0x00];
    }
    return bits | (out_of_range << 63);
}

/* MSE and PEEN as recovered from the reference's README table (SURVEY.md section 6):
 * MSE = sum((x-y)^2)/N, PEEN% = 100*sqrt(sum((x-y)^2)/sum(x^2)); double accumulation. */
void oracle_metrics_u8(const unsigned char *x, const unsigned char *y, size_t n,
                       double *mse, double *peen)
{
    double se = 0.0, e = 0.0;
    for (size_t i = 0; i < n; i++) {
        double d = (double)x[i] - (double)y[i];
        se += d * d;
        e += (double)x[i] * (double)x[i];
    }
    *mse = se / (double)n;
    *peen = e > 0.0 ? 100.0 * sqrt(se / e) : 0.0;
}

void oracle_metrics_f32(const float *x, const float *y, size_t n, double *mse, double *peen)
{
    double se = 0.0, e = 0.0;
    for (size_t i = 0; i < n; i++) {
        double d = (double)x[i] - (double)y[i];
        se += d * d;
        e += (double)x[i] * (double)x[i];
    }
    *mse = se / (double)n;
    *peen = e > 0.0 ? 100.0 * sqrt(se / e) : 0.0;
}

/* FNV-1a-64 over little-endian int32 coefficients / u8 pixels (SURVEY.md Appendix B). */
uint64_t oracle_fnv_coef(const float *coef, size_t n)
{
    uint64_t h = 0xcbf29ce484222325ull;
    for (size_t i = 0; i < n; i++) {
        int32_t v = (int32_t)coef[i];
        for (int b = 0; b < 4; b++) {
            h ^= (uint64_t)((uint32_t)v >> (8 * b)) & 0xff;
            h *= 0x100000001b3ull;
        }
    }
    return h;
}

uint64_t oracle_fnv_u8(const unsigned char *p, size_t n)
{
    uint64_t h = 0xcbf29ce484222325ull;
    for (size_t i = 0; i < n; i++) {
        h ^= p[i];
        h *= 0x100000001b3ull;
    }
    return h;
}

/* Wall-clock seconds of `reps` round trips (best of reps), for the CPU baseline. */
double oracle_time_roundtrip(const float *img, int H, int W, float *out, int reps, int threads)
{
    double best = 1e30;
    for (int i = 0; i < reps; i++) {
        struct timespec a, b;
        clock_gettime(CLOCK_MONOTONIC, &a);
        oracle_roundtrip(img, H, W, k_haweel_T, k_jpeg_Q, ~(uint64_t)0, NULL, out, threads);
        clock_gettime(CLOCK_MONOTONIC, &b);
        double t = (double)(b.tv_sec - a.tv_sec) + 1e-9 * (double)(b.tv_nsec - a.tv_nsec);
        if (t < best) best = t;
    }
    return best;
}

int oracle_max_threads(void)
{
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}
