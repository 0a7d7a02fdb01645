// rgb_kernels.cuh -- interleaved RGB u8 -> YCbCr -> per-plane fused round trip -> RGB u8, ONE pass.
//
// SURVEY.md section 8f "generality: multi-channel / YCbCr with the chroma Q table".  The reference's
// loader returns interleaved RGB for colour files (utils.cu:62-64) and its programs then ignore the
// channel count (main_newAppr.cu:47).  This kernel is the colour version of the same pipeline:
//   RGB -> YCbCr  : libjpeg's jccolor.c fixed point (SCALEBITS 16, FIX(x) = x*65536+0.5, ONE_HALF
//                   rounding, CBCR_OFFSET + ONE_HALF - 1 for Cb/Cr), 8-bit samples, 4:4:4
//   per plane     : the reference's u8 pipeline (convertToFloat utils.cu:10-15 -> dct_all_blocks_cuda
//                   -> idct_all_blocks_cuda -> convertToUnsignedChar utils.cu:18-24), luminance
//                   table for Y, ITU-T T.81 Annex K.2 chrominance table for Cb and Cr
//   YCbCr -> RGB  : libjpeg's jdcolor.c (Cr_r_tab / Cb_b_tab rounded per entry, the two green terms
//                   share one shift).
// One thread owns one 8x8 pixel position in all three planes.  The input is read once (three
// 8-byte loads per row and lane; a warp's row is one contiguous 768-byte span), Y goes straight
// into the transform registers, Cb and Cr wait as bytes in shared memory; every finished plane is
// parked as bytes in shared memory until the last one is done, then the rows are converted back
// and stored.  24 KiB of shared memory per 128-thread CTA, no barrier (every thread only ever
// touches its own slots).  k_rgb_forward and k_rgb_inverse are its two halves, split at the
// zig-zag coefficient streams.
//
// The forward conversion runs on the integer dot-product unit (IDP.2A, see rgb_to_ycc_sums).  The inverse
// conversion's constants need 17 bits, so it runs on the FP32 pipe, exactly: every product and partial sum
// of the libjpeg expressions is an integer of magnitude < 2^24 (e.g. 255 * 65536 + 32768), the
// coefficients are pre-scaled by 2^-16 (a pure exponent shift), so each FMA is exact and
// ">> 16" (arithmetic) is a round-toward-minus-infinity to integer, done by adding 1.5 * 2^23 in
// RM mode.  Both are bit-identical to the integer code (tests/test_gpu_rgb.py against the CPU restatement,
// which is pinned against the real libjpeg).
#pragma once

#include "dct_kernels.cuh"

namespace b200dct {

// ITU-T T.81 Annex K.2
__host__ __device__ constexpr float jpeg_q_chroma(int k)
{
    constexpr float q[64] = {
        17, 18, 24, 47, 99, 99, 99, 99,
        18, 21, 26, 66, 99, 99, 99, 99,
        24, 26, 56, 99, 99, 99, 99, 99,
        47, 66, 99, 99, 99, 99, 99, 99,
        99, 99, 99, 99, 99, 99, 99, 99,
        99, 99, 99, 99, 99, 99, 99, 99,
        99, 99, 99, 99, 99, 99, 99, 99,
        99, 99, 99, 99, 99, 99, 99, 99};
    return q[k];
}
// Quantiser tables of the two plane kinds as {1/Q, Q} pairs: the plane loop below is ONE copy of the
// transform code for Y, Cb and Cr, so the table entries cannot be immediates or fixed constant-bank
// operands; one 64-bit constant load per coefficient fetches both values (-Q is an operand modifier).
struct PlaneTables {
    float2 rd[64];     // {RN(1/Q), Q}
    uint32_t keep[64]; // 0xffffffff kept / 0 dropped
};
struct RgbParams {
    const void *in;  // interleaved RGB u8, 8-byte aligned rows (fused and forward kernels)
    void *out;       // (fused and inverse kernels)
    void *zz;        // three block-major zig-zag int16 streams (Y, Cb, Cr), zz_plane bytes apart: optional output of
                     // the fused kernel, output of the forward kernel, input of the inverse kernel
    size_t in_pitch, out_pitch, zz_plane, zz_pitch; // bytes; zz_pitch = bytes per block-row of one stream
    int bx, by;
    EarlyPath ep;    // not for the fused kernel with streams
    PlaneTables t[2]; // [0] luminance, [1] chrominance
};
template <bool MASKED, bool FASTDIV>
struct QPlane {
    static constexpr bool masked = MASKED;
    static constexpr bool fastdiv = FASTDIV;
    const PlaneTables &t;
    __device__ __forceinline__ explicit QPlane(const PlaneTables &tt) : t(tt) {}
    __device__ __forceinline__ float rcp(int k) const { return t.rd[k].x; }
    __device__ __forceinline__ float d(int k) const { return t.rd[k].y; }
    __device__ __forceinline__ float neg_d(int k) const { return -t.rd[k].y; }
    __device__ __forceinline__ uint32_t keep(int k) const { return t.keep[k]; }
};

constexpr float RGB_MAGIC = 12582912.0f; // 1.5 * 2^23: x + MAGIC in RM mode = MAGIC + floor(x) for |x| < 2^22
#define B200_FIX(x) ((float)((int)((x) * 65536.0 + 0.5)) * (1.0f / 65536.0f))

__device__ __forceinline__ float floor_magic(float x) { return __fadd_rd(x, RGB_MAGIC); } // MAGIC + floor(x)

// ---- RGB -> YCbCr on the integer dot-product unit (IDP.2A: two 16-bit x 8-bit products per instruction).
// libjpeg's expressions are sums of 16-bit constants times 8-bit samples, which is exactly what dp2a computes:
// with the pixel's bytes {R, G, B, x} in one word, .lo multiplies (R, G) and .hi (B, x) by the two halves of the
// constant word.  7 instructions per pixel instead of 6 byte-to-float conversions + 9 FMA + 3 floors; the sample
// is byte 2 of the 32-bit result (every result is in [0, 2^24)).  FIX(0.5) = 32768 does not fit a signed 16-bit
// half, so it travels as an unsigned half next to a zero (Cb) or negated as -32768 (Cr, whose sum is subtracted).
#define B200_IFIX(x) ((int)((x) * 65536.0 + 0.5))
__device__ __forceinline__ uint32_t dp2a_lo_uu(uint32_t a, uint32_t b, uint32_t c) { uint32_t d; asm("dp2a.lo.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c)); return d; }
__device__ __forceinline__ uint32_t dp2a_hi_uu(uint32_t a, uint32_t b, uint32_t c) { uint32_t d; asm("dp2a.hi.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c)); return d; }
__device__ __forceinline__ int dp2a_lo_su(uint32_t a, uint32_t b, int c) { int d; asm("dp2a.lo.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c)); return d; }
__device__ __forceinline__ int dp2a_hi_su(uint32_t a, uint32_t b, int c) { int d; asm("dp2a.hi.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c)); return d; }
__host__ __device__ constexpr uint32_t halves(int lo, int hi) { return ((uint32_t)lo & 0xffffu) | ((uint32_t)hi << 16); }
// pixel word {R, G, B, x} -> the three 32-bit sums whose byte 2 is Y, Cb, Cr (jccolor.c rgb_ycc_convert)
__device__ __forceinline__ void rgb_to_ycc_sums(uint32_t w, uint32_t &y, uint32_t &cb, uint32_t &cr)
{
    constexpr int ONE_HALF = 1 << 15, CBCR = (128 << 16) + ONE_HALF - 1; // CBCR_OFFSET + ONE_HALF - 1
    y = dp2a_hi_uu(halves(B200_IFIX(0.11400), 0), w, dp2a_lo_uu(halves(B200_IFIX(0.29900), B200_IFIX(0.58700)), w, (uint32_t)ONE_HALF));
    cb = dp2a_hi_uu(halves(32768, 0), w, (uint32_t)dp2a_lo_su(halves(-B200_IFIX(0.16874), -B200_IFIX(0.33126)), w, CBCR));
    // Cr = CBCR + 32768 R - FIX(0.41869) G - FIX(0.08131) B = CBCR - (-32768 R + FIX(0.41869) G + FIX(0.08131) B)
    cr = (uint32_t)(CBCR - dp2a_hi_su(halves(B200_IFIX(0.08131), 0), w, dp2a_lo_su(halves(-32768, B200_IFIX(0.41869)), w, 0)));
}
// byte 2 of eight 32-bit sums as eight packed bytes
__device__ __forceinline__ uint2 pack_byte2(const uint32_t (&v)[8])
{
    uint2 o;
    o.x = __byte_perm(__byte_perm(v[0], v[1], 0x0062), __byte_perm(v[2], v[3], 0x0062), 0x5410);
    o.y = __byte_perm(__byte_perm(v[4], v[5], 0x0062), __byte_perm(v[6], v[7], 0x0062), 0x5410);
    return o;
}
// Code size matters here: the L1.5 instruction cache holds 32 KiB, and the first version of this
// kernel (Y transformed by its own copy of the code with immediate tables, both colour conversions
// unrolled over the 8 rows: 5232 instructions = 84 KiB, executed once per thread) spent 5 of 6 issue
// slots waiting for instructions (ncu: stall no_instruction 5.2 per issue, 346 us per 8192^2 image).
// Now the three planes run through ONE copy of the transform in a loop, and the two conversions are
// one row of code each, looped over the rows through shared memory.
// QK: 0 all coefficients kept, exact fast division; 1 mask + exact fast division; 2 mask + __fdiv_rn
constexpr int RGB_CTAS_PER_SM = 5;
// [plane][row][thread] 8-byte slots: a warp's access is 256 contiguous bytes (conflict-free)
using RgbPark = uint2[3][8][128];

// The pieces below are shared by the fused kernel and the two halves of the split API.  Thread 0 of a CTA is always
// inside the image: it is the CTA's leader in the early path (EarlyPath).
// load + RGB -> YCbCr (jccolor.c rgb_ycc_convert) of the thread's 8x8 position, one row per iteration
__device__ __forceinline__ void rgb_load_ycc(const RgbParams &P, long long by, int bxi, int tid, bool early, RgbPark &park)
{
    const char *src = (const char *)P.in + (size_t)by * 8 * P.in_pitch + (size_t)bxi * 24;
#pragma unroll 1
    for (int r = 0; r < 8; r++) {
        const uint2 *row = reinterpret_cast<const uint2 *>(src + (size_t)r * P.in_pitch);
        uint2 a, b, c;
        if (early) a = __ldcg(row), b = __ldcg(row + 1), c = __ldcg(row + 2); // L2 only: never a stale L1 line
        else a = __ldg(row), b = __ldg(row + 1), c = __ldg(row + 2);
        const uint32_t w[6] = {a.x, a.y, b.x, b.y, c.x, c.y};
        // pixel k occupies bytes 3k .. 3k+2 of the 24-byte row: {R, G, B, next byte} as one word (the
        // fourth byte meets a zero constant)
        const uint32_t px[8] = {w[0], __byte_perm(w[0], w[1], 0x6543), __byte_perm(w[1], w[2], 0x5432), w[2] >> 8,
                                w[3], __byte_perm(w[3], w[4], 0x6543), __byte_perm(w[4], w[5], 0x5432), w[5] >> 8};
        uint32_t yv[8], cbv[8], crv[8];
        sfor<8>([&](auto k) { rgb_to_ycc_sums(px[IC(k)], yv[IC(k)], cbv[IC(k)], crv[IC(k)]); });
        park[0][r][tid] = pack_byte2(yv);
        park[1][r][tid] = pack_byte2(cbv);
        park[2][r][tid] = pack_byte2(crv);
    }
}
// YCbCr -> RGB (jdcolor.c ycc_rgb_convert) of eight pixels, each plane's samples as eight packed bytes, stored
// as 24 bytes at `dst` (8-byte aligned)
__device__ __forceinline__ void ycc_row_to_rgb(uint2 yw, uint2 bw, uint2 rw, char *dst)
{
    float o[24];
    sfor<8>([&](auto k) {
        const uint32_t ys = IC(k) < 4 ? yw.x : yw.y, bs = IC(k) < 4 ? bw.x : bw.y, rs = IC(k) < 4 ? rw.x : rw.y;
        const float ym = u8_to_float(ys, IC(k) & 3) - RGB_MAGIC;
        const float cb = u8_shifted(bs, IC(k) & 3), cr = u8_shifted(rs, IC(k) & 3);
        o[3 * IC(k)] = floor_magic(__fmaf_rn(cr, B200_FIX(1.40200), 0.5f)) + ym;
        o[3 * IC(k) + 1] = floor_magic(__fmaf_rn(cr, -B200_FIX(0.71414), __fmaf_rn(cb, -B200_FIX(0.34414), 0.5f))) + ym;
        o[3 * IC(k) + 2] = floor_magic(__fmaf_rn(cb, B200_FIX(1.77200), 0.5f)) + ym;
    });
    uint2 *row = reinterpret_cast<uint2 *>(dst);
    row[0] = make_uint2(pack4_u8(o[0], o[1], o[2], o[3]), pack4_u8(o[4], o[5], o[6], o[7]));       // range_limit = saturation
    row[1] = make_uint2(pack4_u8(o[8], o[9], o[10], o[11]), pack4_u8(o[12], o[13], o[14], o[15]));
    row[2] = make_uint2(pack4_u8(o[16], o[17], o[18], o[19]), pack4_u8(o[20], o[21], o[22], o[23]));
}
// YCbCr -> RGB of the parked planes + store, one row per iteration
__device__ __forceinline__ void rgb_store_ycc(const RgbParams &P, long long by, int bxi, int tid, const RgbPark &park)
{
    char *dst = (char *)P.out + (size_t)by * 8 * P.out_pitch + (size_t)bxi * 24;
#pragma unroll 1
    for (int r = 0; r < 8; r++) ycc_row_to_rgb(park[0][r][tid], park[1][r][tid], park[2][r][tid], dst + (size_t)r * P.out_pitch);
}

// ZZ: also emit the three zig-zag coefficient streams (its own instantiation: 150 instructions the
// default kernel does not have to carry through the instruction cache)
template <int QK, bool FINV, bool ZZ>
__global__ void __launch_bounds__(128, RGB_CTAS_PER_SM) k_rgb(const __grid_constant__ RgbParams P)
{
    __shared__ RgbPark park;
    const int tid = threadIdx.y * 32 + threadIdx.x;
    const int bxi = blockIdx.y * 32 + threadIdx.x;
    const long long by = (long long)blockIdx.x * 4 + threadIdx.y;
    if (bxi >= P.bx || by >= P.by) return;
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    bool early = false;
    if constexpr (!ZZ) early = early_check(P.ep, tid == 0); // the host never offers the early path with streams (written mid-kernel)
    if (!early) asm volatile("griddepcontrol.wait;" ::: "memory");

    rgb_load_ycc(P, by, bxi, tid, early, park);

    // ---- the three planes through one copy of the reference's u8 pipeline
#pragma unroll 1
    for (int plane = 0; plane < 3; plane++) {
        float2 p[8][4];
        sfor<8>([&](auto r) { unpack_u8_shifted(park[plane][IC(r)][tid], p[IC(r)]); }); // convertToFloat + sub_matrix_scalar
        const QPlane<QK != 0, QK != 2> qp(P.t[plane != 0]);
        forward_block<KeepAll>(p, HaweelT<false, true>{}, qp);
        if constexpr (ZZ) st_block_zigzag((char *)P.zz + (size_t)plane * P.zz_plane + (size_t)by * P.zz_pitch + (size_t)bxi * 128, p);
        if constexpr (FINV) {
            inverse_block_fast<true>(p, qp);
        } else {
            inverse_block<KeepAll>(p, HaweelT<true, true>{}, qp);
            sfor<8>([&](auto r) { shift_row(p[IC(r)], 128.0f); }); // add_matrix_scalar, utils_kernels.cu:29
        }
        sfor<8>([&](auto r) { park[plane][IC(r)][tid] = pack_u8_row(p[IC(r)]); }); // convertToUnsignedChar, utils.cu:21
    }

    if (early) asm volatile("griddepcontrol.wait;" ::: "memory"); // every global write waits for the predecessor
    rgb_store_ycc(P, by, bxi, tid, park);
    early_feed(P.ep, tid == 0);
}

// ---- the two halves of k_rgb (b200dct_forward_rgb / b200dct_inverse_rgb): the same arithmetic, so
// inverse(forward(x)) == the fused round trip bit for bit while no stream entry saturates int16.
// Forward: RGB -> YCbCr -> per plane dct + quantise -> zig-zag streams (reads P.in, writes P.zz).  Early
// path: load, colour conversion and the Y transform run before the wait, which precedes the first stream store.
template <int QK>
__global__ void __launch_bounds__(128, RGB_CTAS_PER_SM) k_rgb_forward(const __grid_constant__ RgbParams P)
{
    __shared__ RgbPark park;
    const int tid = threadIdx.y * 32 + threadIdx.x;
    const int bxi = blockIdx.y * 32 + threadIdx.x;
    const long long by = (long long)blockIdx.x * 4 + threadIdx.y;
    if (bxi >= P.bx || by >= P.by) return;
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    const bool early = early_check(P.ep, tid == 0);
    if (!early) asm volatile("griddepcontrol.wait;" ::: "memory");

    rgb_load_ycc(P, by, bxi, tid, early, park);
#pragma unroll 1
    for (int plane = 0; plane < 3; plane++) {
        float2 p[8][4];
        sfor<8>([&](auto r) { unpack_u8_shifted(park[plane][IC(r)][tid], p[IC(r)]); }); // convertToFloat + sub_matrix_scalar
        forward_block<KeepAll>(p, HaweelT<false, true>{}, QPlane<QK != 0, QK != 2>(P.t[plane != 0]));
        if (early && plane == 0) asm volatile("griddepcontrol.wait;" ::: "memory"); // before the first global write
        st_block_zigzag((char *)P.zz + (size_t)plane * P.zz_plane + (size_t)by * P.zz_pitch + (size_t)bxi * 128, p);
    }
    early_feed(P.ep, tid == 0);
}
// Inverse: zig-zag streams -> per plane dequantise + idct + convertToUnsignedChar -> YCbCr -> RGB (reads P.zz,
// writes P.out).  Both inverse routines read only Q (qp.d), never the mask or 1/Q, so there is no quantiser variant.
// Early path: the streams are loaded and transformed before the wait, which precedes the RGB stores.
template <bool FINV>
__global__ void __launch_bounds__(128, RGB_CTAS_PER_SM) k_rgb_inverse(const __grid_constant__ RgbParams P)
{
    __shared__ RgbPark park;
    const int tid = threadIdx.y * 32 + threadIdx.x;
    const int bxi = blockIdx.y * 32 + threadIdx.x;
    const long long by = (long long)blockIdx.x * 4 + threadIdx.y;
    if (bxi >= P.bx || by >= P.by) return;
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    const bool early = early_check(P.ep, tid == 0);
    if (!early) asm volatile("griddepcontrol.wait;" ::: "memory");

#pragma unroll 1
    for (int plane = 0; plane < 3; plane++) {
        float2 p[8][4];
        const char *src = (const char *)P.zz + (size_t)plane * P.zz_plane + (size_t)by * P.zz_pitch + (size_t)bxi * 128;
        if (early) ld_block_zigzag_cg(src, p);
        else ld_block_zigzag(src, p);
        const QPlane<false, true> qp(P.t[plane != 0]);
        if constexpr (FINV) {
            inverse_block_fast<true>(p, qp);
        } else {
            inverse_block<KeepAll>(p, HaweelT<true, true>{}, qp);
            sfor<8>([&](auto r) { shift_row(p[IC(r)], 128.0f); }); // add_matrix_scalar, utils_kernels.cu:29
        }
        sfor<8>([&](auto r) { park[plane][IC(r)][tid] = pack_u8_row(p[IC(r)]); }); // convertToUnsignedChar, utils.cu:21
    }

    if (early) asm volatile("griddepcontrol.wait;" ::: "memory"); // every global write waits for the predecessor
    rgb_store_ycc(P, by, bxi, tid, park);
    early_feed(P.ep, tid == 0);
}

} // namespace b200dct
