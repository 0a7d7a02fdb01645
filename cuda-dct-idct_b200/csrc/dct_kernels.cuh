// dct_kernels.cuh -- the two kernel families built on dct_core.cuh.
//
//   k_direct : one thread per 8x8 block, 128-bit LDG/STG straight from/to HBM.  Works for
//              any H,W multiple of 8 and any aligned pitch; also carries the
//              "input overwritten with X-128" side effect of the reference's dct_*
//              functions (main_newAppr.cu:273) for the compat wrappers.
//   k_tma    : persistent kernel, one CTA per SM.  Every warp runs its own two-buffer
//              pipeline: lane 0 issues a TMA tile load (8 image rows x 32 blocks) into a
//              128B-swizzled shared-memory buffer and all lanes wait on the warp's
//              mbarrier, pull their block into registers with conflict-free LDS.128,
//              immediately re-arm the buffer with the next tile's TMA load, transform in
//              registers, write the result tile to a second swizzled buffer and hand it
//              to a TMA store.  No __syncthreads anywhere; HBM sees only full 1 KiB row
//              segments in both directions.
#pragma once

#include <cuda.h>

#include "dct_core.cuh"

namespace b200dct {

enum { MODE_FWD = 0, MODE_INV = 1, MODE_RT = 2 };
// which transform arithmetic a kernel is compiled for: any dense T as ordered FMA chains, Haweel's
// T as compile-time constants (the reference's chains minus the zero terms), or a dense T with
// symmetric even / antisymmetric odd rows evaluated through its even/odd halves (dct_core.cuh)
enum { TK_DENSE = 0, TK_HAWEEL = 1, TK_DENSE_SYM = 2 };
// DT_I16ZZ: compact coefficient stream, block-major -- block (r, c) of the H/8 x W/8 grid is 64
// consecutive int16 in JPEG zig-zag order at byte offset r*pitch + c*128 (direct family only)
enum { DT_F32 = 0, DT_U8 = 1, DT_I16 = 2, DT_I16ZZ = 3, DT_NONE = -1 };
// quantiser variants: 0 = JPEG immediates, all kept; 1 = parameter tables, fast exact
// division, mask applied; 2 = parameter tables, __fdiv_rn (divisors outside the proven set)
// 3..7 = JPEG immediates with the first 6..10 zig-zag coefficients retained, the mask a
// compile-time constant (README.md:63 of the reference): fused round trips only
enum { Q_IMM = 0, Q_PARAM = 1, Q_PARAM_DIV = 2, Q_IMM_K6 = 3, Q_IMM_K7 = 4, Q_IMM_K8 = 5, Q_IMM_K9 = 6, Q_IMM_K10 = 7 };

struct CommonParams {
    QuantTables q;
    DenseT t;
};

template <int QMODE>
struct QSel { // Q_IMM and Q_IMM_K6..K10
    using type = QImm;
    __device__ __forceinline__ static QImm make(const QuantTables &) { return QImm{}; }
};
template <int QMODE>
struct KeepOf {
    using type = KeepMask<(QMODE >= Q_IMM_K6 && QMODE <= Q_IMM_K10) ? zigzag_prefix_mask(QMODE - Q_IMM_K6 + 6) : ~0ull>;
};
template <>
struct QSel<Q_PARAM> {
    using type = QParam<true, true>;
    __device__ __forceinline__ static type make(const QuantTables &q) { return type(q); }
};
template <>
struct QSel<Q_PARAM_DIV> {
    using type = QParam<true, false>;
    __device__ __forceinline__ static type make(const QuantTables &q) { return type(q); }
};

// Runs the selected stages on a block held in p.
//   FWD: pixels-128 -> C      INV: C -> R      RT: pixels-128 -> (C via emit_coef) -> R
// FINV: the factored (+-1 LSB) inverse of dct_core.cuh instead of the reference's ordered chains;
// it leaves pixels WITH the +128 already added (callers must not add it again).
// Kernels whose inverse leaves the +128 already added: the factored inverse and the symmetric dense T.
__host__ __device__ constexpr bool inverse_is_biased(int tk, bool finv) { return finv || tk == TK_DENSE_SYM; }

template <int MODE, int TK, int QMODE, bool CBANK, bool FINV = false, class EmitCoef>
__device__ __forceinline__ void run_block(float2 (&p)[8][4], const CommonParams &cp, EmitCoef &&emit_coef)
{
    constexpr bool SPARSE = TK == TK_HAWEEL;
    static_assert(!FINV || (SPARSE && MODE != MODE_FWD && KeepOf<QMODE>::type::all), "factored inverse: Haweel's T, runtime masks only");
    auto qp = QSel<QMODE>::make(cp.q);
    // a compile-time mask prunes the forward; the inverse may rely on it only when it consumes
    // the coefficients this very thread produced (fused round trip)
    using KM = typename KeepOf<QMODE>::type;
    static_assert(KM::all || (SPARSE && MODE == MODE_RT), "compile-time masks: sparse fused round trips only");
    if constexpr (MODE != MODE_INV) {
        if constexpr (SPARSE) forward_block<KM>(p, HaweelT<false, CBANK>{}, qp);
        else if constexpr (TK == TK_DENSE_SYM) forward_block_sym(p, cp.t, qp);
        else forward_block(p, RuntimeT<false>(cp.t), qp);
    }
    if constexpr (MODE == MODE_RT) emit_coef(p);
    if constexpr (MODE != MODE_FWD) {
        if constexpr (FINV) inverse_block_fast<true>(p, qp);
        else if constexpr (SPARSE) inverse_block<KM>(p, HaweelT<true, CBANK>{}, qp);
        else if constexpr (TK == TK_DENSE_SYM) inverse_block_sym(p, cp.t, qp);
        else inverse_block(p, RuntimeT<true>(cp.t), qp);
    }
}

// ============================================================== direct family
// the completion counters of the early-load protocol are read past every cache level that could be stale
__device__ __forceinline__ unsigned long long ld_counter(const unsigned long long *p)
{
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
// f32 metrics: every block's float sums are converted EXACTLY to unsigned 128-bit fixed point in units of 2^-50 and
// accumulated as integers (order-independent => deterministic).  The floor: a block sum rounds to a multiple of
// 2^-50; the ceiling: totals below 2^78 (2^22 blocks of 64 pixels of magnitude 2^20 sum to 2^68).
constexpr double METRICS_FIXED_POINT = 0x1p50;
// One metrics accumulator: {sse lo, sse hi, energy lo, energy hi, non-zero count} (64-bit words)
constexpr int MACC_WORDS = 5;
struct U128 {
    unsigned long long lo, hi;
};
__device__ __forceinline__ U128 u128_add(U128 a, U128 b)
{
    U128 r;
    r.lo = a.lo + b.lo;
    r.hi = a.hi + b.hi + (r.lo < a.lo ? 1ull : 0ull);
    return r;
}
__device__ __forceinline__ U128 u128_shfl_xor(U128 a, int o)
{
    return U128{__shfl_xor_sync(0xffffffffu, a.lo, o), __shfl_xor_sync(0xffffffffu, a.hi, o)};
}
// a non-negative finite f32 block sum s -> round(s * 2^50) as 128 bits: s * 2^50 is exact in double, its part above
// 2^64 truncates exactly, the remainder is below 2^64 and holds at most 24 significant bits
__device__ __forceinline__ U128 metrics_fixed(float s)
{
    const double d = (double)s * METRICS_FIXED_POINT;
    const unsigned long long hi = __double2ull_rz(d * 0x1p-64);
    return U128{__double2ull_rn(__fma_rn(-(double)hi, 0x1p64, d)), hi};
}
// adds v to the 128-bit slot {lo, hi} with two 64-bit atomics; the carry out of lo comes from the returned old value,
// so the final pair is the exact sum whatever order the atomics land in
__device__ __forceinline__ void atomic_add_u128(unsigned long long *slot, U128 v)
{
    const unsigned long long old = atomicAdd(&slot[0], v.lo);
    const unsigned long long hi = v.hi + (old + v.lo < old ? 1ull : 0ull);
    if (hi) atomicAdd(&slot[1], hi);
}
// CTA reductions of the metrics kernels: u8 sums stay 64-bit (exact integers far below 2^64), f32 sums are U128
__device__ __forceinline__ unsigned long long acc_add(unsigned long long a, unsigned long long b) { return a + b; }
__device__ __forceinline__ U128 acc_add(U128 a, U128 b) { return u128_add(a, b); }
__device__ __forceinline__ unsigned long long acc_shfl_xor(unsigned long long a, int o) { return __shfl_xor_sync(0xffffffffu, a, o); }
__device__ __forceinline__ U128 acc_shfl_xor(U128 a, int o) { return u128_shfl_xor(a, o); }
__device__ __forceinline__ U128 acc_wide(unsigned long long a) { return U128{a, 0}; }
__device__ __forceinline__ U128 acc_wide(U128 a) { return a; }
__host__ __device__ __forceinline__ double u128_to_double(unsigned long long lo, unsigned long long hi)
{
    return (double)hi * 0x1p64 + (double)lo;
}
constexpr int DIRECT_BATCH_MAX = 64; // images per launch of the batch entry point (1 KiB of kernel parameters)
struct DirectParams {
    const void *in;   // FWD/RT: pixels (PIX dtype); INV: coefficients (coef_dt)
    void *out;        // FWD: coefficients (coef_dt); INV/RT: pixels (PIX dtype)
    void *coef;       // RT only: optional coefficient plane (coef_dt), else NULL
    float *shifted;   // FWD only: optional img-128 write-back (f32), else NULL
    size_t in_pitch, out_pitch, coef_pitch, shifted_pitch; // bytes
    int bx, by;       // blocks per row / block rows
    int coef_dt;      // DT_F32 / DT_I16
    double *partials; // METRICS kernels, two-launch form: 3 doubles per CTA {sum (x-y)^2, sum x^2, non-zero coefficients}
    // METRICS kernels, one-launch form (macc != NULL): every CTA adds its integer sums {sum (x-y)^2, sum x^2} (u8: exact
    // integers; f32: per-block float sums as 128-bit fixed point in units of 2^-50, the TMA family's convention) and its
    // non-zero count to macc[0..MACC_WORDS) with 64-bit atomics (order-independent => deterministic); the last CTA out
    // (mdone[1] counts them) adds the totals, divided by metrics_scale, into acc[0..2] and leaves macc and the counter zeroed
    unsigned long long *macc;
    uint32_t *mdone;
    double *acc;
    double metrics_scale;
    int zz_smem;      // 1: the launch carries ZZ_SMEM_BYTES of dynamic shared memory for the zig-zag stream transpose
    // batch of separately allocated images of one shape (b200dct_roundtrip_batch): image z of the launch
    // is blockIdx.z, its planes come from these tables instead of in / out (pixels only: no coefficient
    // plane, no side effect, no metrics); 0 = the single image above
    int nimg;
    // f32 planes that are 32-byte aligned in address and pitch move with 256-bit accesses: bit 0 = the input plane
    // (all inputs of a batch), bit 1 = the output plane, bit 2 = the optional coefficient plane of a round trip
    int v8;
    // early = E > 0 (never with a coefficient plane beside a round trip, the X-128 write-back or a zig-zag input
    // stream: every global write must be in the store section): the host has established that nothing
    // this launch READS is written by the launch it may overlap with (see early loads, b200dct.cu).  The first
    // E CTAs of the grid (one machine-full: later CTAs only start once these have left, i.e. after the
    // predecessor completed) load their block (L2-coherent loads) and transform it before griddepcontrol.wait,
    // only their stores wait for the predecessor to complete: they work in the slots its last wave leaves idle.
    int early;
    // completion counter of the (device, stream) record (b200dct.cu): chain_feed = F > 0: the last F CTAs of
    // the grid add 1 each at their end; a CTA takes the early path only if the counter still reads below
    // chain_target, i.e. the predecessor is provably still running.  (One reader per CTA, F <= 1024 feeders:
    // 32768 warps polling one L2 line per launch cost the HBM-bound kernels 2-15 us.)
    int chain_feed;
    unsigned long long *chain;
    unsigned long long chain_target;
    const void *img_in[DIRECT_BATCH_MAX];
    void *img_out[DIRECT_BATCH_MAX];
    CommonParams cp;
};
constexpr int ZZ_SMEM_BYTES = 4 * 4096; // one 4 KiB span per warp of the 128-thread CTA

// ---- per-row global accessors (one 8-pixel row of one block) ----
__device__ __forceinline__ void ld_row_f32(const void *base, float2 (&r)[4])
{
    // plain (coherent) loads: the forward kernel may write image-128 back over the very
    // rows it read (the reference's in-place sub_matrix_scalar), which rules out ld.global.nc
    const float4 a = reinterpret_cast<const float4 *>(base)[0];
    const float4 b = reinterpret_cast<const float4 *>(base)[1];
    r[0] = make_float2(a.x, a.y); r[1] = make_float2(a.z, a.w);
    r[2] = make_float2(b.x, b.y); r[3] = make_float2(b.z, b.w);
}
__device__ __forceinline__ void ld_row_f32_cg(const void *base, float2 (&r)[4]) // L2 only: never a stale L1 line
{
    const float4 a = __ldcg(reinterpret_cast<const float4 *>(base));
    const float4 b = __ldcg(reinterpret_cast<const float4 *>(base) + 1);
    r[0] = make_float2(a.x, a.y); r[1] = make_float2(a.z, a.w);
    r[2] = make_float2(b.x, b.y); r[3] = make_float2(b.z, b.w);
}
// 256-bit accesses (sm_100: LDG.E.256 / STG.E.256): a lane's whole 32-byte block row -- one full sector -- per
// instruction instead of two half-sector 128-bit accesses; rows must be 32-byte aligned (P.v8).
template <bool CG>
__device__ __forceinline__ void ld_row_f32_v8(const void *base, float2 (&r)[4])
{
    if constexpr (CG)
        asm volatile("ld.global.cg.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                     : "=f"(r[0].x), "=f"(r[0].y), "=f"(r[1].x), "=f"(r[1].y), "=f"(r[2].x), "=f"(r[2].y), "=f"(r[3].x), "=f"(r[3].y) : "l"(base) : "memory");
    else
        asm volatile("ld.global.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                     : "=f"(r[0].x), "=f"(r[0].y), "=f"(r[1].x), "=f"(r[1].y), "=f"(r[2].x), "=f"(r[2].y), "=f"(r[3].x), "=f"(r[3].y) : "l"(base) : "memory");
}
__device__ __forceinline__ void st_row_f32_v8(void *base, const float2 (&r)[4])
{
    asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(base), "f"(r[0].x), "f"(r[0].y), "f"(r[1].x), "f"(r[1].y),
                 "f"(r[2].x), "f"(r[2].y), "f"(r[3].x), "f"(r[3].y) : "memory");
}
__device__ __forceinline__ void st_row_f32(void *base, const float2 (&r)[4])
{
    reinterpret_cast<float4 *>(base)[0] = make_float4(r[0].x, r[0].y, r[1].x, r[1].y);
    reinterpret_cast<float4 *>(base)[1] = make_float4(r[2].x, r[2].y, r[3].x, r[3].y);
}
__device__ __forceinline__ void unpack_u8_shifted(uint2 w, float2 (&r)[4])
{
    r[0] = make_float2(u8_shifted(w.x, 0), u8_shifted(w.x, 1));
    r[1] = make_float2(u8_shifted(w.x, 2), u8_shifted(w.x, 3));
    r[2] = make_float2(u8_shifted(w.y, 0), u8_shifted(w.y, 1));
    r[3] = make_float2(u8_shifted(w.y, 2), u8_shifted(w.y, 3));
}
__device__ __forceinline__ uint2 pack_u8_plus128(const float2 (&r)[4])
{
    uint2 w;
    w.x = pack4_u8(r[0].x + 128.0f, r[0].y + 128.0f, r[1].x + 128.0f, r[1].y + 128.0f);
    w.y = pack4_u8(r[2].x + 128.0f, r[2].y + 128.0f, r[3].x + 128.0f, r[3].y + 128.0f);
    return w;
}
__device__ __forceinline__ uint2 pack_u8_row(const float2 (&r)[4]) // pixels that already carry the +128
{
    uint2 w;
    w.x = pack4_u8(r[0].x, r[0].y, r[1].x, r[1].y);
    w.y = pack4_u8(r[2].x, r[2].y, r[3].x, r[3].y);
    return w;
}
__device__ __forceinline__ uint4 pack_i16(const float2 (&r)[4])
{
    return make_uint4(pack2_i16(r[0].x, r[0].y), pack2_i16(r[1].x, r[1].y),
                      pack2_i16(r[2].x, r[2].y), pack2_i16(r[3].x, r[3].y));
}
__device__ __forceinline__ void unpack_i16(uint4 w, float2 (&r)[4])
{
    r[0] = make_float2(i16_lo(w.x), i16_hi(w.x)); r[1] = make_float2(i16_lo(w.y), i16_hi(w.y));
    r[2] = make_float2(i16_lo(w.z), i16_hi(w.z)); r[3] = make_float2(i16_lo(w.w), i16_hi(w.w));
}
// block <-> 128 contiguous bytes of zig-zag ordered int16, as 8 chunks of 16 bytes
__device__ __forceinline__ uint32_t smem_u32(const void *p);
__device__ __forceinline__ uint4 lds128u(uint32_t a);
__device__ __forceinline__ void sts128u(uint32_t a, uint4 v);
template <int G>
__device__ __forceinline__ uint4 zigzag_chunk(float2 (&c)[8][4])
{
    uint4 w;
    w.x = pack2_i16(zigzag_elem<8 * G + 0>(c), zigzag_elem<8 * G + 1>(c));
    w.y = pack2_i16(zigzag_elem<8 * G + 2>(c), zigzag_elem<8 * G + 3>(c));
    w.z = pack2_i16(zigzag_elem<8 * G + 4>(c), zigzag_elem<8 * G + 5>(c));
    w.w = pack2_i16(zigzag_elem<8 * G + 6>(c), zigzag_elem<8 * G + 7>(c));
    return w;
}
template <int G>
__device__ __forceinline__ void zigzag_unchunk(uint4 w, float2 (&c)[8][4])
{
    zigzag_elem<8 * G + 0>(c) = i16_lo(w.x); zigzag_elem<8 * G + 1>(c) = i16_hi(w.x);
    zigzag_elem<8 * G + 2>(c) = i16_lo(w.y); zigzag_elem<8 * G + 3>(c) = i16_hi(w.y);
    zigzag_elem<8 * G + 4>(c) = i16_lo(w.z); zigzag_elem<8 * G + 5>(c) = i16_hi(w.z);
    zigzag_elem<8 * G + 6>(c) = i16_lo(w.w); zigzag_elem<8 * G + 7>(c) = i16_hi(w.w);
}
// Per-lane access: 8 x 128-bit, lanes 128 bytes apart (every instruction touches 32 half-used
// sectors).  Used for partial warps at the right edge and when no shared memory was provided.
__device__ __forceinline__ void st_block_zigzag(void *base, float2 (&c)[8][4])
{
    sfor<8>([&](auto g) { reinterpret_cast<uint4 *>(base)[IC(g)] = zigzag_chunk<IC(g)>(c); });
}
__device__ __forceinline__ void ld_block_zigzag(const void *base, float2 (&c)[8][4])
{
    sfor<8>([&](auto g) { zigzag_unchunk<IC(g)>(__ldg(reinterpret_cast<const uint4 *>(base) + IC(g)), c); });
}
__device__ __forceinline__ void ld_block_zigzag_cg(const void *base, float2 (&c)[8][4]) // L2 only: never a stale L1 line
{
    sfor<8>([&](auto g) { zigzag_unchunk<IC(g)>(__ldcg(reinterpret_cast<const uint4 *>(base) + IC(g)), c); });
}
// Cooperative access for a full warp (32 adjacent blocks = one contiguous 4 KiB span): the span
// is transposed through a 4 KiB shared-memory buffer so that every global instruction moves 512
// contiguous bytes.  Chunk c of block b lives at b*128 + ((c ^ (b & 7)) * 16): both the per-block
// side (a quarter-warp = 8 blocks, same c) and the per-span side (a quarter-warp = 8 chunks of
// one block) hit 8 distinct 16-byte bank groups -- conflict-free.
__device__ __forceinline__ uint32_t zigzag_slot(int b, int c) { return (uint32_t)(b * 128 + ((c ^ (b & 7)) * 16)); }
__device__ __forceinline__ void st_warp_zigzag(void *span, uint32_t buf, int lane, float2 (&c)[8][4])
{
    sfor<8>([&](auto g) { sts128u(buf + zigzag_slot(lane, IC(g)), zigzag_chunk<IC(g)>(c)); });
    __syncwarp();
    sfor<8>([&](auto g) {
        reinterpret_cast<uint4 *>(span)[IC(g) * 32 + lane] = lds128u(buf + zigzag_slot(IC(g) * 4 + (lane >> 3), lane & 7));
    });
}
__device__ __forceinline__ void ld_warp_zigzag(const void *span, uint32_t buf, int lane, float2 (&c)[8][4])
{
    sfor<8>([&](auto g) {
        sts128u(buf + zigzag_slot(IC(g) * 4 + (lane >> 3), lane & 7), __ldg(reinterpret_cast<const uint4 *>(span) + IC(g) * 32 + lane));
    });
    __syncwarp();
    sfor<8>([&](auto g) { zigzag_unchunk<IC(g)>(lds128u(buf + zigzag_slot(lane, IC(g))), c); });
}
__device__ __forceinline__ void shift_row(float2 (&r)[4], float s)
{
    sfor<4>([&](auto j) { r[IC(j)] = fadd2(r[IC(j)], bc(s)); });
}

// METRICS (round trip only): the kernel also accumulates, per CTA, the squared error and the
// signal energy between the pixels it read and the pixels it wrote (as stored: u8 after
// clamp+truncate) and the number of non-zero quantised coefficients, and writes them to
// P.partials[cta]; k_reduce_partials then adds them up in a fixed order (deterministic).
// The input row is re-read at the end (an L2 hit) instead of being kept in 64 registers.
// Occupancy of the direct family: 5 CTAs of 128 threads per SM (<= 96 registers, 24-40 bytes of
// spill) instead of the 4 that the unconstrained 128 registers allow.  Same box, 8192^2
// (profiles/r01_direct_occupancy.txt): dense-T round trip 108.2 -> 92.4 us, f32 87.7 -> 85.9,
// u8 65.3 -> 65.3; 6 CTAs (80 registers, up to 400 bytes of spill) loses everywhere.
#ifndef B200DCT_DIRECT_MIN_BLOCKS
#define B200DCT_DIRECT_MIN_BLOCKS 5
#endif
#ifndef B200DCT_METRICS_MIN_BLOCKS
#define B200DCT_METRICS_MIN_BLOCKS 4
#endif
template <int MODE, int TK, int QMODE, int PIX, bool METRICS = false, bool FINV = false>
__global__ void __launch_bounds__(128, METRICS ? B200DCT_METRICS_MIN_BLOCKS : B200DCT_DIRECT_MIN_BLOCKS) k_direct(const __grid_constant__ DirectParams P)
{
    constexpr bool BIASED = inverse_is_biased(TK, FINV);
    // CTA = 32 block-columns x 4 block-rows; grid.x walks block-rows (no 65535 limit),
    // grid.y walks groups of 32 block-columns.  Lanes of a warp are horizontally adjacent
    // blocks, so each row access of a warp covers one contiguous 1 KiB segment.
    static_assert(!METRICS || MODE == MODE_RT, "metrics are defined for the round trip");
    int bxi = blockIdx.y * 32 + threadIdx.x;
    long long by = (long long)blockIdx.x * 4 + threadIdx.y;
    const bool valid = bxi < P.bx && by < P.by;
    if constexpr (!METRICS) {
        if (!valid) return;
    } else if (!valid) { // stay for the CTA reduction; work on block (0,0), store nothing
        bxi = 0;
        by = 0;
    }
    float m_sse = 0.0f, m_en = 0.0f, m_nnz = 0.0f;
    unsigned i_xx = 0, i_xy = 0, i_yy = 0; // u8 metrics
    // programmatic dependent launch (no-ops unless the host asked for it): see k_tma
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    bool early = false;
    if (P.early != 0 && P.coef == nullptr && P.shifted == nullptr && // every global write of such a launch is in its store section
        (blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x < (unsigned)P.early) { // CTA-uniform
        __shared__ int s_early;
        if (threadIdx.x == 0 && threadIdx.y == 0) s_early = ld_counter(P.chain) < P.chain_target; // thread (0,0) is always valid
        __syncthreads();
        early = s_early != 0;
    }
    if (!early) asm volatile("griddepcontrol.wait;" ::: "memory");

    // zig-zag stream: full warps transpose their 4 KiB span through shared memory (warp-uniform)
    extern __shared__ uint8_t zz_raw[];
    const bool zz_coop = P.zz_smem && (int)(blockIdx.y * 32 + 32) <= P.bx;
    const uint32_t zz_buf = smem_u32(zz_raw) + threadIdx.y * 4096;

    float2 p[8][4];
    // ---- load
    // batch launches: the planes of image blockIdx.z (a register-indexed read of the parameter bank,
    // warp-uniform); the output pointer is fetched again at the store so that it is not live in between
    const void *const in_plane = P.nimg ? P.img_in[blockIdx.z] : P.in;
    if constexpr (MODE == MODE_INV) {
        const char *src = (const char *)in_plane + (size_t)by * 8 * P.in_pitch;
        if (P.coef_dt == DT_F32) {
            if ((P.v8 & 1) && early) sfor<8>([&](auto r) { ld_row_f32_v8<true>(src + IC(r) * P.in_pitch + (size_t)bxi * 32, p[IC(r)]); });
            else if (P.v8 & 1) sfor<8>([&](auto r) { ld_row_f32_v8<false>(src + IC(r) * P.in_pitch + (size_t)bxi * 32, p[IC(r)]); });
            else if (early) sfor<8>([&](auto r) { ld_row_f32_cg(src + IC(r) * P.in_pitch + (size_t)bxi * 32, p[IC(r)]); });
            else sfor<8>([&](auto r) { ld_row_f32(src + IC(r) * P.in_pitch + (size_t)bxi * 32, p[IC(r)]); });
        } else if (P.coef_dt == DT_I16ZZ) { // pitch = bytes per block-row of the stream (never on the early path)
            const char *row = (const char *)in_plane + (size_t)by * P.in_pitch;
            if (zz_coop) ld_warp_zigzag(row + (size_t)blockIdx.y * 4096, zz_buf, threadIdx.x, p);
            else ld_block_zigzag(row + (size_t)bxi * 128, p);
        } else {
            uint4 w[8];
            if (early) sfor<8>([&](auto r) { w[IC(r)] = __ldcg(reinterpret_cast<const uint4 *>(src + IC(r) * P.in_pitch + (size_t)bxi * 16)); });
            else sfor<8>([&](auto r) { w[IC(r)] = __ldg(reinterpret_cast<const uint4 *>(src + IC(r) * P.in_pitch + (size_t)bxi * 16)); });
            sfor<8>([&](auto r) { unpack_i16(w[IC(r)], p[IC(r)]); });
        }
    } else if constexpr (PIX == DT_F32) {
        const char *src = (const char *)in_plane + (size_t)by * 8 * P.in_pitch + (size_t)bxi * 32;
        if ((P.v8 & 1) && early) sfor<8>([&](auto r) { ld_row_f32_v8<true>(src + IC(r) * P.in_pitch, p[IC(r)]); });
        else if (P.v8 & 1) sfor<8>([&](auto r) { ld_row_f32_v8<false>(src + IC(r) * P.in_pitch, p[IC(r)]); });
        else if (early) sfor<8>([&](auto r) { ld_row_f32_cg(src + IC(r) * P.in_pitch, p[IC(r)]); });
        else sfor<8>([&](auto r) { ld_row_f32(src + IC(r) * P.in_pitch, p[IC(r)]); });
        sfor<8>([&](auto r) { shift_row(p[IC(r)], -128.0f); }); // sub_matrix_scalar, utils_kernels.cu:16
        if constexpr (MODE == MODE_FWD) {
            if (P.shifted) {
                char *dst = (char *)P.shifted + (size_t)by * 8 * P.shifted_pitch + (size_t)bxi * 32;
                sfor<8>([&](auto r) { st_row_f32(dst + IC(r) * P.shifted_pitch, p[IC(r)]); });
            }
        }
    } else {
        const char *src = (const char *)in_plane + (size_t)by * 8 * P.in_pitch + (size_t)bxi * 8;
        uint2 w[8];
        if (early) sfor<8>([&](auto r) { w[IC(r)] = __ldcg(reinterpret_cast<const uint2 *>(src + IC(r) * P.in_pitch)); });
        else sfor<8>([&](auto r) { w[IC(r)] = __ldg(reinterpret_cast<const uint2 *>(src + IC(r) * P.in_pitch)); });
        sfor<8>([&](auto r) { unpack_u8_shifted(w[IC(r)], p[IC(r)]); });
    }

    auto store_coef = [&](void *plane, size_t pitch, bool v8, float2 (&c)[8][4]) {
        char *dst = (char *)plane + (size_t)by * 8 * pitch;
        if (P.coef_dt == DT_F32) {
            if (v8) sfor<8>([&](auto r) { st_row_f32_v8(dst + IC(r) * pitch + (size_t)bxi * 32, c[IC(r)]); });
            else sfor<8>([&](auto r) { st_row_f32(dst + IC(r) * pitch + (size_t)bxi * 32, c[IC(r)]); });
        } else if (P.coef_dt == DT_I16ZZ) {
            char *row = (char *)plane + (size_t)by * pitch;
            if (zz_coop) st_warp_zigzag(row + (size_t)blockIdx.y * 4096, zz_buf, threadIdx.x, c);
            else st_block_zigzag(row + (size_t)bxi * 128, c);
        } else {
            sfor<8>([&](auto r) {
                *reinterpret_cast<uint4 *>(dst + IC(r) * pitch + (size_t)bxi * 16) = pack_i16(c[IC(r)]);
            });
        }
    };

    run_block<MODE, TK, QMODE, true, FINV>(p, P.cp, [&](float2 (&c)[8][4]) {
        if (P.coef && valid) store_coef(P.coef, P.coef_pitch, (P.v8 & 4) != 0, c);
        if constexpr (METRICS) {
            sfor<8>([&](auto r) {
                sfor<4>([&](auto j) {
                    // coefficients are integer-valued: min(|c|, 1) is 1 for every non-zero one
                    m_nnz += fminf(fabsf(c[IC(r)][IC(j)].x), 1.0f) + fminf(fabsf(c[IC(r)][IC(j)].y), 1.0f);
                });
            });
        }
    });

    // ---- store
    if (early) asm volatile("griddepcontrol.wait;" ::: "memory"); // every global write waits for the predecessor
    void *const out_plane = P.nimg ? P.img_out[blockIdx.z] : P.out;
    if constexpr (MODE == MODE_FWD) {
        store_coef(out_plane, P.out_pitch, (P.v8 & 2) != 0, p);
    } else if constexpr (PIX == DT_F32) {
        char *dst = (char *)out_plane + (size_t)by * 8 * P.out_pitch + (size_t)bxi * 32;
        const char *src = (const char *)P.in + (size_t)by * 8 * P.in_pitch + (size_t)bxi * 32;
        sfor<8>([&](auto r) {
            if constexpr (!BIASED) shift_row(p[IC(r)], 128.0f); // add_matrix_scalar, utils_kernels.cu:29
            if (valid) {
                if (P.v8 & 2) st_row_f32_v8(dst + IC(r) * P.out_pitch, p[IC(r)]);
                else st_row_f32(dst + IC(r) * P.out_pitch, p[IC(r)]);
            }
            if constexpr (METRICS) {
                float2 x[4];
                ld_row_f32(src + IC(r) * P.in_pitch, x);
                sfor<4>([&](auto j) {
                    const float dx = x[IC(j)].x - p[IC(r)][IC(j)].x, dy = x[IC(j)].y - p[IC(r)][IC(j)].y;
                    m_sse = __fmaf_rn(dx, dx, m_sse); m_sse = __fmaf_rn(dy, dy, m_sse);
                    m_en = __fmaf_rn(x[IC(j)].x, x[IC(j)].x, m_en); m_en = __fmaf_rn(x[IC(j)].y, x[IC(j)].y, m_en);
                });
            }
        });
    } else {
        char *dst = (char *)out_plane + (size_t)by * 8 * P.out_pitch + (size_t)bxi * 8;
        const char *src = (const char *)P.in + (size_t)by * 8 * P.in_pitch + (size_t)bxi * 8;
        sfor<8>([&](auto r) {
            const uint2 w = BIASED ? pack_u8_row(p[IC(r)]) : pack_u8_plus128(p[IC(r)]);
            if (valid) *reinterpret_cast<uint2 *>(dst + IC(r) * P.out_pitch) = w;
            if constexpr (METRICS) {
                // integers: sum (x-y)^2 = sum x^2 - 2 sum x*y + sum y^2, four pixels per IDP.4A
                // (64 pixels x 255^2 < 2^23: exact in u32 and, at the end, in float)
                const uint2 xin = __ldg(reinterpret_cast<const uint2 *>(src + IC(r) * P.in_pitch));
                i_xx = __dp4a(xin.x, xin.x, i_xx); i_xx = __dp4a(xin.y, xin.y, i_xx);
                i_xy = __dp4a(xin.x, w.x, i_xy);   i_xy = __dp4a(xin.y, w.y, i_xy);
                i_yy = __dp4a(w.x, w.x, i_yy);     i_yy = __dp4a(w.y, w.y, i_yy);
            }
        });
    }

    if (P.chain_feed && threadIdx.x == 0 && threadIdx.y == 0 &&
        (blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x + (unsigned)P.chain_feed >= gridDim.x * gridDim.y * gridDim.z)
        atomicAdd(P.chain, 1ull); // one of the last CTAs of the grid is (as good as) done
    if constexpr (METRICS) {
        if (P.macc) { // one-launch form
            using Acc = std::conditional_t<PIX == DT_U8, unsigned long long, U128>;
            Acc v[2] = {Acc{}, Acc{}};
            unsigned long long nz = 0;
            if (valid) {
                if constexpr (PIX == DT_U8) {
                    v[0] = i_xx + i_yy - 2u * i_xy;
                    v[1] = i_xx;
                } else {
                    v[0] = metrics_fixed(m_sse);
                    v[1] = metrics_fixed(m_en);
                }
                nz = (unsigned long long)m_nnz;
            }
            __shared__ Acc ired[2][4];
            __shared__ unsigned long long inz[4];
            const int lane = threadIdx.x, w = threadIdx.y;
            for (int o = 16; o > 0; o >>= 1) {
                v[0] = acc_add(v[0], acc_shfl_xor(v[0], o));
                v[1] = acc_add(v[1], acc_shfl_xor(v[1], o));
                nz += __shfl_xor_sync(0xffffffffu, nz, o);
            }
            if (lane == 0) {
                ired[0][w] = v[0];
                ired[1][w] = v[1];
                inz[w] = nz;
            }
            __syncthreads();
            if (w == 0 && lane == 0) {
                sfor<2>([&](auto q) {
                    atomic_add_u128(&P.macc[2 * IC(q)], acc_wide(acc_add(acc_add(ired[IC(q)][0], ired[IC(q)][1]), acc_add(ired[IC(q)][2], ired[IC(q)][3]))));
                });
                atomicAdd(&P.macc[4], (inz[0] + inz[1]) + (inz[2] + inz[3]));
                __threadfence();
                if (atomicAdd(&P.mdone[1], 1u) == gridDim.x * gridDim.y - 1u) { // every other CTA's sums are in
                    __threadfence();
                    unsigned long long t[MACC_WORDS];
                    sfor<MACC_WORDS>([&](auto q) { t[IC(q)] = atomicExch(&P.macc[IC(q)], 0ull); });
                    P.acc[0] += u128_to_double(t[0], t[1]) / P.metrics_scale;
                    P.acc[1] += u128_to_double(t[2], t[3]) / P.metrics_scale;
                    P.acc[2] += (double)t[4];
                    P.mdone[1] = 0;
                    __threadfence();
                }
            }
            return;
        }
        if constexpr (PIX == DT_U8) {
            m_sse = (float)(i_xx + i_yy - 2u * i_xy);
            m_en = (float)i_xx;
        }
        double v[3] = {valid ? (double)m_sse : 0.0, valid ? (double)m_en : 0.0, valid ? (double)m_nnz : 0.0};
        __shared__ double red[3][4];
        const int lane = threadIdx.x, w = threadIdx.y;
        sfor<3>([&](auto q) {
            for (int o = 16; o > 0; o >>= 1) v[IC(q)] += __shfl_xor_sync(0xffffffffu, v[IC(q)], o);
            if (lane == 0) red[IC(q)][w] = v[IC(q)];
        });
        __syncthreads();
        if (w == 0 && lane < 3) {
            const size_t cta = (size_t)blockIdx.y * gridDim.x + blockIdx.x;
            P.partials[cta * 3 + lane] = (red[lane][0] + red[lane][1]) + (red[lane][2] + red[lane][3]);
        }
    }
}

// Resident CTAs per SM of one instantiation (cached): the host needs it to decide whether a launch
// has more CTAs than the machine holds at once (early loads of its successor, b200dct.cu).
template <void (*KERNEL)(DirectParams)>
inline int direct_ctas_per_sm(size_t smem)
{
    static int cached[2] = {-1, -1};
    int &v = cached[smem ? 1 : 0];
    if (v < 0) {
        int n = 0;
        v = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, KERNEL, 128, smem) == cudaSuccess ? n : 0;
    }
    return v;
}

// ============================================================== TMA family
// Tile = 8 image rows x 32 blocks (256 pixels).  Shared-memory images of a tile:
//   f32 : 8 KiB, rows of 1 KiB = 8 segments of 128 B, hardware SWIZZLE_128B: the 16-byte
//         chunk c of segment s sits at chunk c^s.  Lane l owns segment l>>2, chunks
//         2(l&3), 2(l&3)+1, so a quarter-warp's LDS.128/STS.128 covers 8 distinct chunk
//         positions: conflict-free (an unswizzled 32-byte lane stride is 2-way).
//   u8  : 2 KiB, rows of 256 B, lane l owns bytes 8l..8l+7 (LDS.64, conflict-free).
//   i16 : 4 KiB, rows of 512 B, lane l owns bytes 16l..16l+15 (LDS.128, conflict-free).
struct TmaParams {
    CUtensorMap in_map;   // FWD/RT: pixels; INV: coefficients
    CUtensorMap out_map;  // FWD: coefficients; INV/RT: pixels
    CUtensorMap coef_map; // RT with coefficient output
    uint32_t tiles_x;     // tiles per tile-row
    uint32_t ntiles;
    int coef_dt;          // DT_F32 / DT_I16
    int has_coef;         // RT: also emit the coefficient plane
    // Dynamic tile scheduler: {next ticket, finished warps}, both 0 at launch and reset to 0
    // by the last warp to leave; NULL = static round-robin (used under stream capture).
    uint32_t *sched;
    uint32_t run;         // tiles per ticket for the first run_tickets tickets, then 1
    uint32_t run_tickets;
    uint32_t buf_bytes;   // size of one tile buffer: the largest tile image among the planes of this call
    // METRICS kernels: {sum (x-y)^2, sum x^2} as 128-bit fixed point in units of 2^-50 and the number of
    // non-zero coefficients (MACC_WORDS words), accumulated with 64-bit integer atomics (order-independent
    // => deterministic)
    unsigned long long *macc;
    double *acc;          // METRICS with the dynamic scheduler: the last warp out adds macc into acc[0..2] and re-zeroes macc
    // 1: the host has established that nothing this launch READS is written by the launch it may
    // overlap with (see early_loads_ok in b200dct.cu): tile loads start before griddepcontrol.wait,
    // every global write (TMA stores, metrics atomics) still waits for the predecessor to complete
    int early_loads;
    // completion counter of the (device, stream) record: chain_feed = 1: the last warp out adds 1; early_loads = 1:
    // a warp only loads early if the counter still reads below chain_target (predecessor provably still running)
    int chain_feed;
    unsigned long long *chain;
    unsigned long long chain_target;
    uint32_t bx;          // blocks per image row (lanes of a right-edge tile beyond it hold TMA zero fill, not pixels)
    CommonParams cp;
};

// every warp owns two tile buffers (in, out) of P.buf_bytes each: 8 KiB when an f32 plane is
// involved, 4 KiB for i16, 2 KiB for an all-u8 round trip
__host__ __device__ constexpr uint32_t tile_bytes_of(int dt) { return dt == DT_F32 ? 8192u : (dt == DT_I16 ? 4096u : 2048u); }

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(bar), "r"(parity) : "memory");
}
// f32 tiles use the 3-d view {32 floats, W/32 segments, H rows}; u8/i16 tiles the 2-d view.
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap *map, uint32_t bar, int c0, int c1, int c2)
{
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap *map, uint32_t bar, int c0, int c1)
{
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap *map, uint32_t src, int c0, int c1, int c2)
{
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
                 ::"l"(map), "r"(src), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap *map, uint32_t src, int c0, int c1)
{
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                 ::"l"(map), "r"(src), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ float4 lds128(uint32_t a)
{
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts128(uint32_t a, float4 v)
{
    asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(a), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ uint4 lds128u(uint32_t a)
{
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts128u(uint32_t a, uint4 v)
{
    asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(a), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ uint2 lds64u(uint32_t a)
{
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts64u(uint32_t a, uint2 v)
{
    asm volatile("st.shared.v2.u32 [%0], {%1,%2};" ::"r"(a), "r"(v.x), "r"(v.y) : "memory");
}

// Swizzled f32 tile accessors.  off0 = byte offset of the lane's first 16-byte chunk in a
// tile row; the second chunk is off0 ^ 16.
__device__ __forceinline__ uint32_t f32_tile_off0(int lane)
{
    return (uint32_t)((lane >> 2) * 128 + (((2 * (lane & 3)) ^ (lane >> 2)) & 7) * 16);
}
__device__ __forceinline__ void tile_ld_f32(uint32_t buf, uint32_t off0, float2 (&p)[8][4])
{
    sfor<8>([&](auto r) {
        const float4 a = lds128(buf + IC(r) * 1024 + off0);
        const float4 b = lds128(buf + IC(r) * 1024 + (off0 ^ 16u));
        p[IC(r)][0] = make_float2(a.x, a.y); p[IC(r)][1] = make_float2(a.z, a.w);
        p[IC(r)][2] = make_float2(b.x, b.y); p[IC(r)][3] = make_float2(b.z, b.w);
    });
}
__device__ __forceinline__ void tile_st_f32(uint32_t buf, uint32_t off0, const float2 (&p)[8][4])
{
    sfor<8>([&](auto r) {
        sts128(buf + IC(r) * 1024 + off0, make_float4(p[IC(r)][0].x, p[IC(r)][0].y, p[IC(r)][1].x, p[IC(r)][1].y));
        sts128(buf + IC(r) * 1024 + (off0 ^ 16u), make_float4(p[IC(r)][2].x, p[IC(r)][2].y, p[IC(r)][3].x, p[IC(r)][3].y));
    });
}

template <int DT>
__device__ __forceinline__ uint32_t tile_bytes()
{
    return tile_bytes_of(DT);
}

// Register budget of the persistent kernel: one CTA per SM, CTA size per kernel flavour.
//  * sparse T, f32 pixels (HBM-bound): 256 threads, <= 255 registers.  Measured on B200 at 8192^2
//    (profiles/r01_tma_warps_sweep.txt): 4 warps 119 us, 6: 96, 7: 90, 8: 84.0, 9: 84.0.  8 warps =
//    2 per scheduler is enough because every thread carries 64 independent FMA chains.  (With
//    single-tile tickets more warps, or a working set above ~1 GiB, collapsed to 113-118 us: the
//    TMA path's address translation thrashes when every SM touches every 2 MiB page; runs of 2
//    consecutive tiles per ticket removed that -- profiles/r01_tma_run_scheduler.txt.)
//  * u8 pixels and dense T (FP32-pipe bound): more, smaller warps -- 512 threads / 128 registers
//    for u8 (tile buffers are only 2 KiB), 384 threads / 168 registers for dense T.
#ifndef B200DCT_TMA_CTA_THREADS
#define B200DCT_TMA_CTA_THREADS 256
#endif
#ifndef B200DCT_TMA_CTA_THREADS_U8
#define B200DCT_TMA_CTA_THREADS_U8 512
#endif
#ifndef B200DCT_TMA_CTA_THREADS_DENSE
#define B200DCT_TMA_CTA_THREADS_DENSE 384
#endif
#ifndef B200DCT_TMA_CTA_THREADS_SYM
#define B200DCT_TMA_CTA_THREADS_SYM 384
#endif
#ifndef B200DCT_TMA_DEFAULT_WARPS
#define B200DCT_TMA_DEFAULT_WARPS 8
#endif
__host__ __device__ constexpr int tma_cta_threads(int pix, int tk)
{
    return pix == DT_U8 ? B200DCT_TMA_CTA_THREADS_U8
                        : (tk == TK_HAWEEL ? B200DCT_TMA_CTA_THREADS : (tk == TK_DENSE_SYM ? B200DCT_TMA_CTA_THREADS_SYM : B200DCT_TMA_CTA_THREADS_DENSE));
}
// the metrics flavour carries three tile buffers per warp (24 KiB): nine warps fill the 227 KiB
#ifndef B200DCT_TMA_CTA_THREADS_METRICS
#define B200DCT_TMA_CTA_THREADS_METRICS 288
#endif
#define B200DCT_TMA_BOUNDS __launch_bounds__(METRICS ? B200DCT_TMA_CTA_THREADS_METRICS : tma_cta_threads(PIX, TK), 1)

// METRICS (f32 round trips): the warp keeps TWO input buffers (the tile being transformed stays in
// shared memory until its output exists, while the next tile is already arriving in the other one),
// so the squared error and the signal energy are taken from the input tile where it already is
// instead of re-reading it from global memory as the direct family's metrics kernel does.
template <int MODE, int TK, int QMODE, int PIX, bool FINV = false, bool METRICS = false>
__global__ void B200DCT_TMA_BOUNDS k_tma(const __grid_constant__ TmaParams P)
{
    static_assert(!METRICS || (MODE == MODE_RT && PIX == DT_F32), "fused metrics on the TMA family: f32 round trips");
    constexpr bool BIASED = inverse_is_biased(TK, FINV);
    constexpr uint32_t NIN = METRICS ? 2u : 1u; // input buffers per warp
    extern __shared__ uint8_t smem_raw[];
    // 1 KiB alignment: the 128B swizzle pattern is a function of address bits 7..9
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nwarps = blockDim.x >> 5;
    const uint32_t in_buf0 = smem_base + warp * (NIN + 1) * P.buf_bytes;
    const uint32_t out_buf = in_buf0 + NIN * P.buf_bytes;
    const uint32_t bar0 = smem_base + nwarps * (NIN + 1) * P.buf_bytes + warp * 8 * NIN;
    uint32_t in_buf = in_buf0, bar = bar0; // METRICS: alternate between the two buffers / barriers
    const uint32_t off0 = f32_tile_off0(lane);

    // Dynamic tile scheduler.  The two dies / far and near L2 slices make SMs progress at
    // different speeds: with a static split the slow SMs set the kernel time while the fast
    // ones idle (17 % of the SM-cycles in ncu, round 1).  Warps therefore draw tickets from
    // a global counter (one atomicAdd per claim, fetched one tile ahead so its latency hides
    // behind the TMA wait).  The first P.run_tickets tickets are worth a RUN of P.run
    // consecutive tiles each (consecutive tiles share their image rows, hence their 2 MiB
    // pages: the TMA unit's address translation is what collapses when every SM wanders
    // over every page of a multi-GiB working set); the remaining tickets are worth one tile
    // each, so the tail of the kernel stays one tile long.  Without a counter (stream
    // capture): static round-robin.
    const uint32_t stride = gridDim.x * nwarps;
    uint32_t *const sched = P.sched;
    uint32_t run_left = 0; // lane 0: tiles still owned after the current one
    auto ticket_tile = [&](uint32_t t) -> uint32_t { // lane 0 only; first tile of ticket t (>= ntiles: none)
        if (t < P.run_tickets) { run_left = P.run - 1; return t * P.run; }
        run_left = 0;
        return P.run_tickets * P.run + (t - P.run_tickets); // may be >= ntiles: the losing ticket
    };
    auto claim_next = [&](uint32_t cur) -> uint32_t { // lane 0 only; returns the next tile
        if (!sched) return cur + stride;
        if (run_left) { run_left--; return cur + 1; }
        return ticket_tile(atomicAdd(&sched[0], 1u) + stride);
    };
    // the first `stride` tickets are pre-assigned (warp-major, CTA-minor) so that no atomic
    // round trip sits in front of the first TMA load; the counter hands out the rest
    uint32_t tile = 0;
    if (lane == 0) tile = sched ? ticket_tile(warp * gridDim.x + blockIdx.x) : warp * gridDim.x + blockIdx.x;
    tile = __shfl_sync(0xffffffffu, tile, 0);
    const bool in_is_f32 = (MODE == MODE_INV) ? (P.coef_dt == DT_F32) : (PIX == DT_F32);
    const uint32_t in_bytes = (MODE == MODE_INV) ? (P.coef_dt == DT_F32 ? 8192u : 4096u) : tile_bytes<PIX>();

    auto issue_load_to = [&](uint32_t t, uint32_t buf, uint32_t b) {
        const int ty = (int)(t / P.tiles_x), tx = (int)(t - (uint32_t)ty * P.tiles_x);
        mbar_expect_tx(b, in_bytes);
        if (in_is_f32) tma_load_3d(buf, &P.in_map, b, 0, tx * 8, ty * 8);
        else tma_load_2d(buf, &P.in_map, b, tx * 256, ty * 8);
    };
    auto issue_load = [&](uint32_t t) { issue_load_to(t, in_buf, bar); };

    // Programmatic dependent launch (only when the host asked for it; no-ops otherwise): let
    // the next kernel in the stream take this SM the moment this CTA leaves it, and do not
    // touch global memory before every earlier kernel has completed and flushed.
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    // early loads: ONE thread of the CTA reads the completion counter (1184 warps polling one L2 line cost
    // 0.5 us per launch); issued here, consumed after the barrier set-up below
    unsigned long long chain_seen = 0;
    if (P.early_loads && threadIdx.x == 0) chain_seen = ld_counter(P.chain);
    if (lane == 0) {
        mbar_init(bar0, 1);
        if constexpr (METRICS) mbar_init(bar0 + 8, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
#ifndef B200DCT_NO_TMAP_PREFETCH
        // the descriptors are kernel parameters, not data of the previous kernel: fetch them into
        // the TMA unit's cache while this CTA still waits for its predecessor (A/B on B200:
        // 82.6 us either way at 8192^2 -- kept because it is free)
        if (warp == 0) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(&P.in_map) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(&P.out_map) : "memory");
            if (P.has_coef) asm volatile("prefetch.tensormap [%0];" ::"l"(&P.coef_map) : "memory");
        }
#endif
    }
    // Only lane 0 ever touches global memory (TMA loads / stores, scheduler and metrics atomics).
    bool early = false;
    if (P.early_loads) { // CTA-uniform; the only CTA-wide barrier of the kernel, before any work exists
        __shared__ int s_early;
        if (threadIdx.x == 0) s_early = chain_seen < P.chain_target;
        __syncthreads();
        early = s_early != 0;
    }
    bool dep_done = !early;
    auto ensure_dep = [&]() { // lane 0, before its first global write
        if (!dep_done) {
            asm volatile("griddepcontrol.wait;" ::: "memory");
            dep_done = true;
        }
    };
    if (!early) asm volatile("griddepcontrol.wait;" ::: "memory");
    if (lane == 0 && tile < P.ntiles) issue_load(tile);
    __syncwarp();

    uint32_t parity = 0;   // METRICS: bit b = parity of barrier b
    uint32_t cur = 0;      // METRICS: which input buffer holds the current tile
    U128 m_sse = {0, 0}, m_en = {0, 0};
    unsigned long long m_nnz = 0;
    while (tile < P.ntiles) {
        const int ty = (int)(tile / P.tiles_x), tx = (int)(tile - (uint32_t)ty * P.tiles_x);
        uint32_t next_l0 = 0;
        if (lane == 0) next_l0 = claim_next(tile);
        uint32_t next_m = 0;
        if constexpr (METRICS) {
            // the other buffer was read for the last time at the end of the previous iteration: the
            // next tile can start arriving before this one is even waited for
            next_m = __shfl_sync(0xffffffffu, next_l0, 0);
            if (lane == 0 && next_m < P.ntiles) issue_load_to(next_m, in_buf0 + (cur ^ 1u) * P.buf_bytes, bar0 + (cur ^ 1u) * 8);
            in_buf = in_buf0 + cur * P.buf_bytes;
            bar = bar0 + cur * 8;
            mbar_wait(bar, (parity >> cur) & 1u);
            parity ^= 1u << cur;
        } else {
            mbar_wait(bar, parity);
            parity ^= 1;
        }

        float2 p[8][4];
        // ---- shared -> registers
        if constexpr (MODE == MODE_INV) {
            if (P.coef_dt == DT_F32) tile_ld_f32(in_buf, off0, p);
            else sfor<8>([&](auto r) { unpack_i16(lds128u(in_buf + IC(r) * 512 + lane * 16), p[IC(r)]); });
        } else if constexpr (PIX == DT_F32) {
            tile_ld_f32(in_buf, off0, p);
            sfor<8>([&](auto r) { shift_row(p[IC(r)], -128.0f); });
        } else {
            sfor<8>([&](auto r) { unpack_u8_shifted(lds64u(in_buf + IC(r) * 256 + lane * 8), p[IC(r)]); });
        }
        // every lane has consumed its part of in_buf: re-arm it with the next tile
        uint32_t next;
        if constexpr (METRICS) {
            next = next_m;
        } else {
            next = __shfl_sync(0xffffffffu, next_l0, 0); // also the warp-wide sync
            if (lane == 0 && next < P.ntiles) issue_load(next);
        }

        auto put_coef_tile = [&](const CUtensorMap *map, float2 (&c)[8][4]) {
            if (lane == 0) tma_store_wait_read(); // previous store has drained out_buf
            __syncwarp();
            if (P.coef_dt == DT_F32) tile_st_f32(out_buf, off0, c);
            else sfor<8>([&](auto r) { sts128u(out_buf + IC(r) * 512 + lane * 16, pack_i16(c[IC(r)])); });
            fence_async_smem();
            __syncwarp();
            if (lane == 0) {
                ensure_dep();
                if (P.coef_dt == DT_F32) tma_store_3d(map, out_buf, 0, tx * 8, ty * 8);
                else tma_store_2d(map, out_buf, tx * 256, ty * 8);
                tma_store_commit();
            }
        };

        float t_nnz = 0.0f;
        run_block<MODE, TK, QMODE, true, FINV>(p, P.cp, [&](float2 (&c)[8][4]) {
            if (P.has_coef) put_coef_tile(&P.coef_map, c);
            if constexpr (METRICS) {
                sfor<8>([&](auto r) {
                    sfor<4>([&](auto j) { // coefficients are integer-valued: min(|c|, 1) counts the non-zero ones
                        t_nnz += fminf(fabsf(c[IC(r)][IC(j)].x), 1.0f) + fminf(fabsf(c[IC(r)][IC(j)].y), 1.0f);
                    });
                });
            }
        });

        // ---- registers -> shared -> HBM
        if constexpr (MODE == MODE_FWD) {
            put_coef_tile(&P.out_map, p);
        } else {
            if (lane == 0) tma_store_wait_read();
            __syncwarp();
            if constexpr (PIX == DT_F32) {
                if constexpr (!BIASED) sfor<8>([&](auto r) { shift_row(p[IC(r)], 128.0f); });
                tile_st_f32(out_buf, off0, p);
                if constexpr (METRICS) {
                    // the pixels as stored against the pixels as read (still in this warp's input buffer)
                    float t_sse = 0.0f, t_en = 0.0f;
                    sfor<8>([&](auto r) {
                        const float4 a = lds128(in_buf + IC(r) * 1024 + off0), b = lds128(in_buf + IC(r) * 1024 + (off0 ^ 16u));
                        const float x[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
                        sfor<4>([&](auto j) {
                            const float dx = x[2 * IC(j)] - p[IC(r)][IC(j)].x, dy = x[2 * IC(j) + 1] - p[IC(r)][IC(j)].y;
                            t_sse = __fmaf_rn(dx, dx, t_sse); t_sse = __fmaf_rn(dy, dy, t_sse);
                            t_en = __fmaf_rn(x[2 * IC(j)], x[2 * IC(j)], t_en); t_en = __fmaf_rn(x[2 * IC(j) + 1], x[2 * IC(j) + 1], t_en);
                        });
                    });
                    // per-block sums (fixed order) -> 128-bit fixed point: integer accumulation is order-independent
                    if ((uint32_t)tx * 32u + (uint32_t)lane < P.bx) {
                        m_sse = u128_add(m_sse, metrics_fixed(t_sse));
                        m_en = u128_add(m_en, metrics_fixed(t_en));
                        m_nnz += (unsigned long long)t_nnz;
                    }
                }
            } else {
                sfor<8>([&](auto r) { sts64u(out_buf + IC(r) * 256 + lane * 8, BIASED ? pack_u8_row(p[IC(r)]) : pack_u8_plus128(p[IC(r)])); });
            }
            fence_async_smem();
            __syncwarp();
            if (lane == 0) {
                ensure_dep();
                if constexpr (PIX == DT_F32) tma_store_3d(&P.out_map, out_buf, 0, tx * 8, ty * 8);
                else tma_store_2d(&P.out_map, out_buf, tx * 256, ty * 8);
                tma_store_commit();
            }
        }
        tile = next;
        if constexpr (METRICS) cur ^= 1u;
    }
    if constexpr (METRICS) {
        for (int o = 16; o > 0; o >>= 1) {
            m_sse = u128_add(m_sse, u128_shfl_xor(m_sse, o));
            m_en = u128_add(m_en, u128_shfl_xor(m_en, o));
            m_nnz += __shfl_xor_sync(0xffffffffu, m_nnz, o);
        }
        if (lane == 0) {
            ensure_dep();
            atomic_add_u128(&P.macc[0], m_sse);
            atomic_add_u128(&P.macc[2], m_en);
            atomicAdd(&P.macc[4], m_nnz);
        }
    }
    if (lane == 0) {
        ensure_dep(); // a warp without tiles must not let the grid finish ahead of its predecessor's flush
        tma_store_wait_read();
        if (sched) {
            // every warp ends on exactly one losing ticket; the last warp out re-zeroes both counters
            __threadfence();
            if (atomicAdd(&sched[1], 1u) == stride - 1) {
                if constexpr (METRICS) {
                    if (P.acc) { // every other warp's sums are in (its atomics precede its fence + ticket)
                        __threadfence();
                        unsigned long long t[MACC_WORDS];
                        sfor<MACC_WORDS>([&](auto q) { t[IC(q)] = atomicExch(&P.macc[IC(q)], 0ull); });
                        P.acc[0] += u128_to_double(t[0], t[1]) / METRICS_FIXED_POINT;
                        P.acc[1] += u128_to_double(t[2], t[3]) / METRICS_FIXED_POINT;
                        P.acc[2] += (double)t[4];
                    }
                }
                sched[0] = 0;
                sched[1] = 0;
                if (P.chain_feed) atomicAdd(P.chain, 1ull); // this launch is (as good as) complete
                __threadfence();
            }
        }
    }
}

} // namespace b200dct
