// rgb420_kernels.cuh -- 4:2:0 chroma subsampling on the split colour path: interleaved RGB u8 -> Y at full
// resolution and Cb, Cr at half resolution in both directions -> three zig-zag coefficient streams, and back.
//
// What libjpeg computes, by default, and therefore what these kernels compute bit for bit (pinned against
// libjpeg-turbo through tests/golden/libjpeg_420.npz):
//   down (jcsample.c h2v2_downsample, no smoothing): a half-resolution sample is (a + b + c + d + bias) >> 2 over
//        its 2x2 group of full-resolution 8-bit Cb or Cr samples (jccolor.c); bias 1 at even output columns and 2
//        at odd ones.
//   up   (jdsample.c h2v2_fancy_upsample): with the half-resolution plane c edge-replicated on all four sides,
//        colsum[x] = 3 c[y][x] + c[y -+ 1][x] (the row above for the upper output row of a pair, the row below
//        for the lower one); the left output pixel of column x is (3 colsum[x] + colsum[x - 1] + 8) >> 4, the
//        right one (3 colsum[x] + colsum[x + 1] + 7) >> 4.
// Per plane the transforms are the 4:4:4 kernels' (convertToFloat, dct, quantise; dequantise, idct,
// convertToUnsignedChar) with the luminance table for Y and the chrominance table for Cb and Cr, through ONE
// copy of the transform code in a loop (see the instruction-cache note in rgb_kernels.cuh).
#pragma once

#include "rgb_kernels.cuh"

namespace b200dct {

struct Rgb420Params {
    const void *in;           // interleaved RGB u8, 8-byte aligned rows (forward kernel)
    void *out;                // (inverse kernel)
    void *zz[3];              // block-major zig-zag int16 streams: Y (H/8 x W/8 blocks), Cb, Cr (H/16 x W/16 blocks each)
    size_t in_pitch, out_pitch;
    size_t zz_pitch[2];       // bytes per block-row: [0] Y, [1] Cb and Cr
    int mx, my;               // MCUs (16 x 16 pixels) per row / column
    EarlyPath ep;
    PlaneTables t[2];         // [0] luminance, [1] chrominance
};

// ---- forward.  A 128-thread CTA covers 16 x 2 MCUs; a thread loads the 8 x 8 pixels of one Y block (as the 4:4:4
// kernel does) and downsamples their Cb and Cr to the 4 x 4 quadrant of its MCU's chroma blocks.  After one barrier
// the CTA's 128 Y blocks and 64 chroma blocks run through one transform loop (threads 0..63 take a second block).
// 12 KiB of shared memory.  Early path: loads, colour conversion and downsampling before the wait; each thread
// waits before its first stream store.
template <int QK>
__global__ void __launch_bounds__(128, RGB_CTAS_PER_SM) k_rgb420_forward(const __grid_constant__ Rgb420Params P)
{
    __shared__ uint2 ypark[8][128];  // [row][thread]
    __shared__ uint2 cpark[2][8][32]; // [Cb / Cr][row][MCU of the CTA]: a warp's access is contiguous
    const int tid = threadIdx.y * 32 + threadIdx.x;
    const int bxi = blockIdx.y * 32 + threadIdx.x;
    const long long by = (long long)blockIdx.x * 4 + threadIdx.y;
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    const bool early = early_check(P.ep, tid == 0);
    if (!early) asm volatile("griddepcontrol.wait;" ::: "memory");

    if (bxi < 2 * P.mx && by < 2 * P.my) {
        const int m = (threadIdx.y >> 1) * 16 + (threadIdx.x >> 1), qx = threadIdx.x & 1, qy = threadIdx.y & 1;
        const char *src = (const char *)P.in + (size_t)by * 8 * P.in_pitch + (size_t)bxi * 24;
#pragma unroll 1
        for (int rp = 0; rp < 4; rp++) { // a pair of pixel rows = one row of the quadrant
            uint32_t hs[2][4];           // Cb, Cr: sums of the 2 x 2 groups
            sfor<2>([&](auto h) {
                const int r = 2 * rp + IC(h);
                const uint2 *row = reinterpret_cast<const uint2 *>(src + (size_t)r * P.in_pitch);
                uint2 a, b, c;
                if (early) a = __ldcg(row), b = __ldcg(row + 1), c = __ldcg(row + 2); // L2 only: never a stale L1 line
                else a = __ldg(row), b = __ldg(row + 1), c = __ldg(row + 2);
                const uint32_t w[6] = {a.x, a.y, b.x, b.y, c.x, c.y};
                const uint32_t px[8] = {w[0], __byte_perm(w[0], w[1], 0x6543), __byte_perm(w[1], w[2], 0x5432), w[2] >> 8,
                                        w[3], __byte_perm(w[3], w[4], 0x6543), __byte_perm(w[4], w[5], 0x5432), w[5] >> 8};
                uint32_t yv[8], cbv[8], crv[8];
                sfor<8>([&](auto k) { rgb_to_ycc_sums(px[IC(k)], yv[IC(k)], cbv[IC(k)], crv[IC(k)]); });
                ypark[r][tid] = pack_byte2(yv);
                sfor<4>([&](auto i) { // the 8-bit samples (byte 2 of each sum) are what libjpeg downsamples
                    const uint32_t sb = __byte_perm(cbv[2 * IC(i)], 0, 0x4442) + __byte_perm(cbv[2 * IC(i) + 1], 0, 0x4442);
                    const uint32_t sr = __byte_perm(crv[2 * IC(i)], 0, 0x4442) + __byte_perm(crv[2 * IC(i) + 1], 0, 0x4442);
                    if constexpr (IC(h) == 0) hs[0][IC(i)] = sb, hs[1][IC(i)] = sr;
                    else hs[0][IC(i)] += sb, hs[1][IC(i)] += sr;
                });
            });
            uint32_t wb = 0, wr = 0; // output column parity = i parity: bias 1, 2, 1, 2
            sfor<4>([&](auto i) {
                wb |= ((hs[0][IC(i)] + 1 + (IC(i) & 1)) >> 2) << (8 * IC(i));
                wr |= ((hs[1][IC(i)] + 1 + (IC(i) & 1)) >> 2) << (8 * IC(i));
            });
            reinterpret_cast<uint32_t *>(&cpark[0][qy * 4 + rp][m])[qx] = wb;
            reinterpret_cast<uint32_t *>(&cpark[1][qy * 4 + rp][m])[qx] = wr;
        }
    }
    __syncthreads();

    bool waited = !early;
#pragma unroll 1
    for (int j = tid; j < 192; j += 128) { // 0..127: the Y block of thread j; then the 32 Cb and the 32 Cr blocks
        const bool luma = j < 128;
        const int c = j - 128, pl = luma ? 0 : 1 + (c >> 5);
        const long long row = luma ? (long long)blockIdx.x * 4 + (j >> 5) : (long long)blockIdx.x * 2 + ((c >> 4) & 1);
        const int col = luma ? blockIdx.y * 32 + (j & 31) : blockIdx.y * 16 + (c & 15);
        if (row >= (luma ? 2LL * P.my : (long long)P.my) || col >= (luma ? 2 * P.mx : P.mx)) continue;
        float2 p[8][4];
        sfor<8>([&](auto r) { unpack_u8_shifted(luma ? ypark[IC(r)][j] : cpark[pl - 1][IC(r)][c & 31], p[IC(r)]); });
        forward_block<KeepAll>(p, HaweelT<false, true>{}, QPlane<QK != 0, QK != 2>(P.t[!luma]));
        if (!waited) { // before the thread's first global write
            asm volatile("griddepcontrol.wait;" ::: "memory");
            waited = true;
        }
        st_block_zigzag((char *)P.zz[pl] + (size_t)row * P.zz_pitch[!luma] + (size_t)col * 128, p);
    }
    early_feed(P.ep, tid == 0);
}

// ---- inverse.  A 128-thread CTA owns a tile of R420_MX x R420_MY MCUs.  Upsampling reads one chroma sample beyond
// the tile on every side, so the CTA also decodes the ring of neighbouring chroma blocks (the same routine as its
// own blocks, hence the same bytes) and parks its own decoded Cb / Cr samples plus that one-sample halo in shared
// memory; at the image border the reads are clamped instead (edge replication), with no extra decode.  One barrier,
// then each thread decodes Y blocks and, row by row, upsamples, converts and stores.  32 x 4 MCUs: 768 own blocks
// (512 Y + 256 chroma) and at most 152 halo chroma blocks, 20 % more transforms; 26 KiB of shared memory.
// Early path: every load and transform before the wait; each thread waits before its first RGB store.
constexpr int R420_MX = 32, R420_MY = 4;
constexpr int R420_CW = R420_MX * 8 + 16; // bytes per parked chroma row: halo sample at 7, own samples from 8, halo after them
constexpr int R420_CH = R420_MY * 8 + 2;  // parked rows: halo row 0, own rows 1 .. R420_MY * 8, halo row after them
constexpr int R420_RING = (R420_MX + 2) * (R420_MY + 2); // chroma blocks of one plane a CTA may decode

// dequantise + idct + convertToUnsignedChar of one block: the same routine for own and ring blocks
template <bool FINV>
__device__ __forceinline__ void inverse_u8_block(const char *src, bool early, const PlaneTables &t, uint2 (&w)[8])
{
    float2 p[8][4];
    if (early) ld_block_zigzag_cg(src, p);
    else ld_block_zigzag(src, p);
    const QPlane<false, true> qp(t);
    if constexpr (FINV) {
        inverse_block_fast<true>(p, qp);
    } else {
        inverse_block<KeepAll>(p, HaweelT<true, true>{}, qp);
        sfor<8>([&](auto r) { shift_row(p[IC(r)], 128.0f); }); // add_matrix_scalar, utils_kernels.cu:29
    }
    sfor<8>([&](auto r) { w[IC(r)] = pack_u8_row(p[IC(r)]); }); // convertToUnsignedChar, utils.cu:21
}

// four chroma samples at columns lx .. lx + 3 of parked row `up` (weight 3) and `nb` (weight 1), with the
// columns left (lx - 1, or lx at the image's left edge) and right -> eight upsampled samples as packed bytes
__device__ __forceinline__ uint2 upsample_h2v2(const unsigned char *up, const unsigned char *nb, int lx, int left, int right)
{
    const uint32_t a = *reinterpret_cast<const uint32_t *>(up + lx), b = *reinterpret_cast<const uint32_t *>(nb + lx);
    int cs[6]; // colsum at columns lx - 1 .. lx + 4
    cs[0] = 3 * up[left] + nb[left];
    cs[5] = 3 * up[right] + nb[right];
    sfor<4>([&](auto k) { cs[1 + IC(k)] = 3 * (int)((a >> (8 * IC(k))) & 0xff) + (int)((b >> (8 * IC(k))) & 0xff); });
    uint32_t o[2] = {0, 0};
    sfor<4>([&](auto k) {
        const uint32_t l = (uint32_t)(3 * cs[1 + IC(k)] + cs[IC(k)] + 8) >> 4, r = (uint32_t)(3 * cs[1 + IC(k)] + cs[2 + IC(k)] + 7) >> 4;
        o[IC(k) >> 1] |= (l | (r << 8)) << (16 * (IC(k) & 1));
    });
    return make_uint2(o[0], o[1]);
}

template <bool FINV>
__global__ void __launch_bounds__(128, RGB_CTAS_PER_SM) k_rgb420_inverse(const __grid_constant__ Rgb420Params P)
{
    __shared__ __align__(16) unsigned char cs[2][R420_CH][R420_CW];
    __shared__ uint2 ypark[8][128];
    const int tid = threadIdx.y * 32 + threadIdx.x;
    const int cy0 = blockIdx.x * R420_MY, cx0 = blockIdx.y * R420_MX; // tile origin, in MCUs = chroma blocks
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    const bool early = early_check(P.ep, tid == 0);
    if (!early) asm volatile("griddepcontrol.wait;" ::: "memory");

    // own chroma blocks and the ring around them: local block (lr, lc), -1 and R420_MY / R420_MX = ring
#pragma unroll 1
    for (int j = tid; j < 2 * R420_RING; j += 128) {
        const int pl = j >= R420_RING, k = j - pl * R420_RING;
        const int lr = k / (R420_MX + 2) - 1, lc = k % (R420_MX + 2) - 1;
        const int gr = cy0 + lr, gc = cx0 + lc;
        if (gr < 0 || gc < 0 || gr >= P.my || gc >= P.mx) continue;
        uint2 w[8];
        inverse_u8_block<FINV>((const char *)P.zz[1 + pl] + (size_t)gr * P.zz_pitch[1] + (size_t)gc * 128, early, P.t[1], w);
        sfor<8>([&](auto r) {
            const int L = 1 + lr * 8 + IC(r); // only the one-sample halo of a ring block is parked
            if (L < 0 || L >= R420_CH) return;
            if (lc < 0) cs[pl][L][7] = (unsigned char)(w[IC(r)].y >> 24);                // its right column
            else if (lc >= R420_MX) cs[pl][L][8 + R420_MX * 8] = (unsigned char)w[IC(r)].x; // its left column
            else *reinterpret_cast<uint2 *>(&cs[pl][L][8 + lc * 8]) = w[IC(r)];
        });
    }
    __syncthreads();

    const int Hc = P.my * 8, Wc = P.mx * 8; // chroma plane size in samples
    bool waited = !early;
#pragma unroll 1
    for (int j = tid; j < R420_MX * R420_MY * 4; j += 128) { // the tile's Y blocks, 2 R420_MX per row
        const int ybr = j / (2 * R420_MX), ybc = j % (2 * R420_MX);
        const int gyr = 2 * cy0 + ybr, gyc = 2 * cx0 + ybc;
        if (gyr >= 2 * P.my || gyc >= 2 * P.mx) continue;
        uint2 w[8];
        inverse_u8_block<FINV>((const char *)P.zz[0] + (size_t)gyr * P.zz_pitch[0] + (size_t)gyc * 128, early, P.t[0], w);
        sfor<8>([&](auto r) { ypark[IC(r)][tid] = w[IC(r)]; });
        if (!waited) { // every global write waits for the predecessor
            asm volatile("griddepcontrol.wait;" ::: "memory");
            waited = true;
        }
        const int x0 = gyc * 4, lx = 8 + ybc * 4;                      // first chroma column under the block
        const int left = x0 == 0 ? lx : lx - 1, right = x0 + 4 == Wc ? lx + 3 : lx + 4;
        char *dst = (char *)P.out + (size_t)gyr * 8 * P.out_pitch + (size_t)gyc * 24;
#pragma unroll 1
        for (int r = 0; r < 8; r++) {
            const int y = gyr * 8 + r, yc = y >> 1;                     // pixel row, chroma row
            const int nb = (y & 1) ? min(yc + 1, Hc - 1) : max(yc - 1, 0);
            const int lu = yc - cy0 * 8 + 1, ln = nb - cy0 * 8 + 1;
            const uint2 bw = upsample_h2v2(cs[0][lu], cs[0][ln], lx, left, right);
            const uint2 rw = upsample_h2v2(cs[1][lu], cs[1][ln], lx, left, right);
            ycc_row_to_rgb(ypark[r][tid], bw, rw, dst + (size_t)r * P.out_pitch);
        }
    }
    early_feed(P.ep, tid == 0);
}

} // namespace b200dct
