// any_kernels.cuh -- fused round trip of images whose sides need not be multiples of 8 and whose rows
// need not be aligned (b200dct_roundtrip_any): k_any (f32, staged through shared memory) and k_any_u8
// (8-bit, word-packed).  Instantiated by inst_any_*.cu only.
#pragma once

#include "dct_kernels.cuh"

namespace b200dct {

// ============================================================== any size, any alignment
// Fused round trip of an image whose sides need not be multiples of 8 and whose rows need not be
// aligned (SURVEY.md section 8f "generality"; the reference silently computes garbage there,
// main_newAppr.cu:261-262): ONE pass, no scratch image.  Blocks that stick out over the right or
// bottom edge are completed by edge replication (coordinates clamped to the last pixel, the same
// values np.pad(mode="edge") produces) and only their inside part is stored.
// Rows are only element-aligned, so accesses are scalar -- but coalesced: a warp owns 8 rows x 256
// pixels (its 32 blocks), moves every row with 8 instructions of 32 consecutive elements, and
// re-shapes rows <-> blocks through an 8 KiB shared-memory stage.  In-place calls are safe: a
// warp reads all of its own region (and nothing else) before it writes it.
struct AnyParams {
    const void *in;
    void *out;
    size_t in_pitch, out_pitch; // bytes, any value >= W * element size
    int H, W;
    CommonParams cp;
};

template <int TK, int QMODE, int PIX, bool FINV = false>
__global__ void __launch_bounds__(128, 5) k_any(const __grid_constant__ AnyParams P)
{
    static_assert(PIX == DT_F32, "8-bit images take k_any_u8");
    constexpr bool BIASED = inverse_is_biased(TK, FINV);
    __shared__ __align__(16) uint32_t stage[4][8 * 256];
    const int lane = threadIdx.x;
    const long long y0 = ((long long)blockIdx.x * 4 + threadIdx.y) * 8;
    if (y0 >= P.H) return; // warp-uniform; lanes whose block lies outside the image stay for the row moves
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    // (No early path across launch boundaries here: it needs L2-only loads, and this kernel lives on the L1 --
    // a warp's 128-byte row pieces are misaligned, neighbouring instructions share their boundary sectors:
    // ld.global.cg measured 104.4 us at 8191^2 against 95.1, more than the 4 us the early path gives back.)
    asm volatile("griddepcontrol.wait;" ::: "memory");
    uint32_t *st = stage[threadIdx.y];
    const int xw = blockIdx.y * 256 + lane;
    // Stage layout: a row is 64 chunks of 16 bytes; chunk c sits at c ^ ((c >> 3) & 1).  The row moves (32
    // consecutive words per instruction) stay permutations of one 128-byte segment, and the block accesses
    // (lane l owns chunks 2l, 2l+1 -- a 32-byte lane stride, 2-way conflicts in a plain layout: ncu counted
    // 12.9 M shared-memory wavefronts against 8.4 M ideal) become conflict-free: lanes 4..7 of every
    // quarter-warp simply take their two chunks in the other order.
    const int lane_odd = lane ^ 4;                         // word index of this lane in the odd 32-word segments
    const int blk_a = lane * 8 + (((lane >> 2) & 1) ? 4 : 0); // word offsets of this lane's two chunks
    const int blk_b = lane * 8 + (((lane >> 2) & 1) ? 0 : 4);

    // rows -> stage (pixels - 128 as float), coordinates clamped to the image
    int xs[8];
    sfor<8>([&](auto s) { xs[IC(s)] = xw + 32 * IC(s) < P.W ? xw + 32 * IC(s) : P.W - 1; });
    sfor<8>([&](auto r) {
        const long long y = y0 + IC(r) < P.H ? y0 + IC(r) : P.H - 1;
        const float *row = reinterpret_cast<const float *>((const char *)P.in + (size_t)y * P.in_pitch);
        sfor<8>([&](auto s) { st[IC(r) * 256 + 32 * IC(s) + ((IC(s) & 1) ? lane_odd : lane)] = __float_as_uint((float)row[xs[IC(s)]] - 128.0f); });
    });
    __syncwarp();
    float2 p[8][4];
    sfor<8>([&](auto r) {
        const float4 a = *reinterpret_cast<const float4 *>(st + IC(r) * 256 + blk_a);
        const float4 b = *reinterpret_cast<const float4 *>(st + IC(r) * 256 + blk_b);
        p[IC(r)][0] = make_float2(a.x, a.y); p[IC(r)][1] = make_float2(a.z, a.w);
        p[IC(r)][2] = make_float2(b.x, b.y); p[IC(r)][3] = make_float2(b.z, b.w);
    });
    __syncwarp(); // every lane has its block: the stage can take the results

    run_block<MODE_RT, TK, QMODE, true, FINV>(p, P.cp, [](float2 (&)[8][4]) {});

    // blocks -> stage: the final pixel value per pixel
    auto fin = [](float v) -> uint32_t { return __float_as_uint(BIASED ? v : v + 128.0f); }; // add_matrix_scalar, utils_kernels.cu:29
    sfor<8>([&](auto r) {
        *reinterpret_cast<uint4 *>(st + IC(r) * 256 + blk_a) =
            make_uint4(fin(p[IC(r)][0].x), fin(p[IC(r)][0].y), fin(p[IC(r)][1].x), fin(p[IC(r)][1].y));
        *reinterpret_cast<uint4 *>(st + IC(r) * 256 + blk_b) =
            make_uint4(fin(p[IC(r)][2].x), fin(p[IC(r)][2].y), fin(p[IC(r)][3].x), fin(p[IC(r)][3].y));
    });
    __syncwarp();
    sfor<8>([&](auto r) {
        if (y0 + IC(r) < P.H) {
            float *row = reinterpret_cast<float *>((char *)P.out + (size_t)(y0 + IC(r)) * P.out_pitch);
            sfor<8>([&](auto s) {
                if (xw + 32 * IC(s) < P.W) row[xw + 32 * IC(s)] = __uint_as_float(st[IC(r) * 256 + 32 * IC(s) + ((IC(s) & 1) ? lane_odd : lane)]);
            });
        }
    });
}

// ---- 8-bit images of any size and alignment: no shared-memory stage at all.
// Byte-aligned rows still consist of aligned 32-bit words: a lane fetches the three aligned words
// that cover its block's 8-byte row and funnel-shifts its own 8 bytes out of them (3 LDG.32 + 2
// SHF per row instead of 8 one-byte loads, conversions and a trip through shared memory), and on
// the way out re-aligns with its left neighbour's last bytes (one SHFL + two SHF) so that almost
// every store is an aligned 32-bit word; only the bytes at the two ends of a warp's 256-pixel span
// and ragged blocks at the right image edge move as single bytes.  Bytes of neighbouring spans
// that ride along in a loaded word are shifted out unused (so concurrent in-place updates of
// them by other warps are harmless) and are never written.  Rows beyond the bottom edge and
// pixels beyond the right edge replicate the last row / pixel (np.pad(mode="edge")).
// 8191^2: 125 us with the staged kernel above -> see profiles/r02_any_size.txt.
// explicit global-space accesses: addresses formed by masking pointer bits lose their address space
// (the compiler falls back to generic LD/ST otherwise)
__device__ __forceinline__ uint32_t ldg_u32(uintptr_t a)
{
    uint32_t v;
    asm volatile("ld.global.u32 %0, [%1];" : "=r"(v) : "l"(a));
    return v;
}
// predicated form: lanes with p == false issue no access at all (and get 0)
__device__ __forceinline__ uint32_t ldg_u32_if(uintptr_t a, bool p)
{
    uint32_t v;
    asm volatile("{\n.reg .pred q;\nsetp.ne.u32 q, %2, 0;\nmov.u32 %0, 0;\n@q ld.global.u32 %0, [%1];\n}" : "=r"(v) : "l"(a), "r"((uint32_t)p));
    return v;
}
__device__ __forceinline__ uint32_t ldg_u8(uintptr_t a)
{
    uint32_t v;
    asm volatile("ld.global.u8 %0, [%1];" : "=r"(v) : "l"(a));
    return v;
}
__device__ __forceinline__ void stg_u32(uintptr_t a, uint32_t v) { asm volatile("st.global.u32 [%0], %1;" ::"l"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void stg_u8(uintptr_t a, uint32_t v) { asm volatile("st.global.u8 [%0], %1;" ::"l"(a), "r"(v) : "memory"); }

template <int TK, int QMODE, bool FINV>
__global__ void __launch_bounds__(128, 5) k_any_u8(const __grid_constant__ AnyParams P)
{
    constexpr bool BIASED = inverse_is_biased(TK, FINV);
    const int lane = threadIdx.x;
    const long long y0 = ((long long)blockIdx.x * 4 + threadIdx.y) * 8;
    if (y0 >= P.H) return; // warp-uniform
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
    const int xb = blockIdx.y * 256 + lane * 8;       // first pixel of this lane's block
    const bool full = xb + 8 <= P.W;                  // the whole block row lies inside the image
    const bool partial = !full && xb < P.W;
    const bool any_partial = __any_sync(0xffffffffu, partial); // at most one lane, in the last span of a row

    // All loads of the block are issued before anything waits for one of them: the main path is
    // branch-free (a per-row branch, even a warp-uniform one, keeps ptxas from hoisting the next
    // row's loads over it -- measured: 8 serialised memory round trips per warp, 101 us at 8191^2).
    // Lanes without a whole block inside the image issue no access (predicated loads, not branches).
    float2 p[8][4];
    uint2 w[8];
    const uintptr_t in0 = (uintptr_t)P.in;
    sfor<8>([&](auto r) {
        const long long y = y0 + IC(r) < P.H ? y0 + IC(r) : P.H - 1;
        const uintptr_t a = in0 + (size_t)y * P.in_pitch + (size_t)xb;
        const uintptr_t wa = a & ~(uintptr_t)3;
        const unsigned sh = (unsigned)(a & 3) * 8;
        const uint32_t w0 = ldg_u32_if(wa, full), w1 = ldg_u32_if(wa + 4, full);
        const uint32_t w2 = ldg_u32_if(wa + (sh ? 8 : 4), full); // the third word holds own bytes iff sh != 0; never read past them
        w[IC(r)].x = __funnelshift_r(w0, w1, sh);
        w[IC(r)].y = __funnelshift_r(w1, w2, sh);
    });
    if (any_partial) { // ragged block at the right edge: one lane of the last span of a row, byte by byte
        if (partial) {
            sfor<8>([&](auto r) {
                const long long y = y0 + IC(r) < P.H ? y0 + IC(r) : P.H - 1;
                const uintptr_t a = in0 + (size_t)y * P.in_pitch + (size_t)xb;
                uint2 v = make_uint2(0u, 0u);
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    const uint32_t b = ldg_u8(a + (xb + k < P.W ? k : P.W - 1 - xb));
                    if (k < 4) v.x |= b << (8 * k);
                    else v.y |= b << (8 * (k - 4));
                }
                w[IC(r)] = v;
            });
        }
    }
    sfor<8>([&](auto r) { unpack_u8_shifted(w[IC(r)], p[IC(r)]); });

    run_block<MODE_RT, TK, QMODE, true, FINV>(p, P.cp, [](float2 (&)[8][4]) {});

    const bool lead = lane == 0;                                                    // nobody to my left in this warp
    const bool trail = !(__shfl_down_sync(0xffffffffu, (int)full, 1) && lane < 31); // nobody to my right completes my last word
    const uintptr_t out0 = (uintptr_t)P.out + (size_t)xb;
    sfor<8>([&](auto r) {
        const uint2 o = BIASED ? pack_u8_row(p[IC(r)]) : pack_u8_plus128(p[IC(r)]);
        w[IC(r)] = o;
        const uint32_t left_hi = __shfl_up_sync(0xffffffffu, o.y, 1); // the left neighbour's last four bytes
        const bool row_ok = y0 + IC(r) < P.H;                         // warp-uniform
        const uintptr_t d = out0 + (size_t)(y0 + IC(r)) * P.out_pitch;
        const unsigned so = (unsigned)(d & 3);                        // warp-uniform
        const uintptr_t q = d & ~(uintptr_t)3;
        const unsigned s = so * 8;
        const bool st = full && row_ok;
        // aligned words: [neighbour's last so bytes | my first 4-so] and [my bytes 4-so .. 8-so); so == 0: my two words
        if (st && (!lead || so == 0)) stg_u32(q, __funnelshift_l(left_hi, o.x, s));
        if (st) stg_u32(q + 4, __funnelshift_l(o.x, o.y, s));
        // the ends of the warp's span: single bytes
        if (st && lead && so != 0) stg_u8(d, o.x);
        if (st && lead && so != 0 && so < 3) stg_u8(d + 1, o.x >> 8);
        if (st && lead && so == 1) stg_u8(d + 2, o.x >> 16);
        if (st && trail && so != 0) stg_u8(d + 7, o.y >> 24);
        if (st && trail && so > 1) stg_u8(d + 6, o.y >> 16);
        if (st && trail && so > 2) stg_u8(d + 5, o.y >> 8);
    });
    if (any_partial) {
        if (partial) {
            sfor<8>([&](auto r) {
                if (y0 + IC(r) < P.H) {
                    const uintptr_t d = out0 + (size_t)(y0 + IC(r)) * P.out_pitch;
#pragma unroll
                    for (int k = 0; k < 8; k++)
                        if (xb + k < P.W) stg_u8(d + k, (k < 4 ? w[IC(r)].x : w[IC(r)].y) >> (8 * (k & 3)));
                }
            });
        }
    }
}

} // namespace b200dct
