// dct_core.cuh -- register-resident 8x8 block transform core for sm_100a.
//
// One thread owns one 8x8 block as 32 packed float pairs (p[row][pair], pair j holds
// columns 2j and 2j+1).  Both separable passes, the quantiser and the dequantiser run
// on registers only: no shared memory, no shuffles, no barriers between the passes.
//
// Arithmetic contract (what makes the quantised coefficients bit-exact against the
// reference kernels, see DESIGN.md "Arithmetic"):
//   * every inner product is the reference's ordered chain of fused multiply-adds,
//     summation index ascending, accumulator starting at +0.0f
//     (cuda_matrix_dct main_newAppr.cu:193-197,206-209; cuda_matrix_idct :236-239,246-248;
//      the same chains in cuda_matrix_dct_paper main_fastAppr.cu:203-227).  Terms whose
//     T entry is exactly 0 are skipped: fma(0,x,s)==s bit-for-bit for finite x because
//     the running sum is never -0.0f.
//   * two independent chains are issued per instruction with Blackwell's packed
//     fma.rn.f32x2 (SASS FFMA2); each half is an IEEE fma.rn, so packing changes
//     nothing numerically.  In the column pass the two halves are adjacent columns and
//     the T entry is a broadcast immediate; in the row pass the two halves are two
//     output columns with the same sparsity pattern and the input is a broadcast
//     register.
//   * quantisation is a correctly rounded division (divide_matrices,
//     utils_kernels.cu:42, PTX div.rn.f32) followed by round-half-away-from-zero.
//     With a known divisor d and r = RN(1/d) the quotient is obtained with three FMAs
//     (q0 = x*r; e = fma(-d,q0,x); q = fma(e,r,q0)), which is the correctly rounded
//     x/d (Markstein); tests/test_gpu_div.py sweeps all 2^32 inputs per divisor.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <type_traits>
#include <utility>

namespace b200dct {

// ---------------------------------------------------------------- static loops
template <class F, int... I>
__device__ __forceinline__ void sfor_impl(F &f, std::integer_sequence<int, I...>)
{
    (f(std::integral_constant<int, I>{}), ...);
}
template <int N, class F>
__device__ __forceinline__ void sfor(F &&f)
{
    sfor_impl(f, std::make_integer_sequence<int, N>{});
}
#define IC(v) (decltype(v)::value)

// ---------------------------------------------------------------- packed fp32
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c)
{
    unsigned long long ra = *reinterpret_cast<unsigned long long *>(&a);
    unsigned long long rb = *reinterpret_cast<unsigned long long *>(&b);
    unsigned long long rc = *reinterpret_cast<unsigned long long *>(&c);
    unsigned long long rd;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rb), "l"(rc));
    return *reinterpret_cast<float2 *>(&rd);
}
__device__ __forceinline__ float2 fadd2(float2 a, float2 b)
{
    unsigned long long ra = *reinterpret_cast<unsigned long long *>(&a);
    unsigned long long rb = *reinterpret_cast<unsigned long long *>(&b);
    unsigned long long rd;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(rd) : "l"(ra), "l"(rb));
    return *reinterpret_cast<float2 *>(&rd);
}
__device__ __forceinline__ float2 fmul2(float2 a, float2 b)
{
    unsigned long long ra = *reinterpret_cast<unsigned long long *>(&a);
    unsigned long long rb = *reinterpret_cast<unsigned long long *>(&b);
    unsigned long long rd;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(rd) : "l"(ra), "l"(rb));
    return *reinterpret_cast<float2 *>(&rd);
}
__device__ __forceinline__ float2 fsub2(float2 a, float2 b)
{
    unsigned long long ra = *reinterpret_cast<unsigned long long *>(&a);
    unsigned long long rb = *reinterpret_cast<unsigned long long *>(&b);
    unsigned long long rd;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(rd) : "l"(ra), "l"(rb));
    return *reinterpret_cast<float2 *>(&rd);
}
__device__ __forceinline__ float2 bc(float v) { return make_float2(v, v); }

// ---------------------------------------------------------------- constants
// Haweel's matrix, spelled exactly as the reference does (double literals narrowed to
// float, main_newAppr.cu:73-81) so that the bit patterns are the reference's.
__host__ __device__ constexpr float haweel(int r, int c)
{
    constexpr float a = (float)0.35355339, h = (float)0.5, p = (float)0.4472136,
                    q = (float)0.2236068, s = (float)0.70710678;
    constexpr float t[64] = {
        a, a, a, a, a, a, a, a,
        h, h, 0, 0, 0, 0, -h, -h,
        p, q, -q, -p, -p, -q, q, p,
        0, 0, -s, 0, 0, s, 0, 0,
        a, -a, -a, a, a, -a, -a, a,
        h, -h, 0, 0, 0, 0, h, -h,
        q, -p, p, -q, -q, p, -p, q,
        0, 0, 0, -s, s, 0, 0, 0};
    return t[r * 8 + c];
}

// JPEG luminance table (main_newAppr.cu:60-68).
__host__ __device__ constexpr float jpeg_q(int k)
{
    constexpr float q[64] = {
        16, 11, 10, 16, 24, 40, 51, 61,
        12, 12, 14, 19, 26, 58, 60, 55,
        14, 13, 16, 24, 40, 57, 69, 56,
        14, 17, 22, 29, 51, 87, 80, 62,
        18, 22, 37, 56, 68, 109, 103, 77,
        24, 35, 55, 64, 81, 104, 113, 92,
        49, 64, 78, 87, 103, 121, 120, 101,
        72, 92, 95, 98, 112, 100, 103, 99};
    return q[k];
}

// Runtime tables handed to the kernels by value (they live in the kernel-parameter
// constant bank, so every use is a c[0x0][..] operand, not a load).
struct QuantTables {
    float neg_d[64];   // -Q
    float rcp[64];     // RN(1/Q)
    float d[64];       //  Q (dequantiser, and divisor of the exact-division fallback)
    uint32_t keep[64]; // 0xffffffff kept / 0 dropped
};
struct DenseT {
    float t[64];  // T[r][c]
    float tt[64]; // T^T, so that {T[x][i],T[x+1][i]} is one aligned 8-byte constant
    // symmetric kernels (rows 2i symmetric, rows 2i+1 antisymmetric, e.g. the true DCT-II):
    // eo[i*4+n] = {T[2i][n], T[2i+1][n]} for n < 4 -- the halves of a packed instruction are an
    // even (symmetric) and an odd (antisymmetric) basis function
    float2 eo[16];
};

// ---------------------------------------------------------------- transform policies
// A policy answers "coefficient multiplying input i in the chain of output a".
//   forward  column pass: M[y][x] = sum_i T[y][i] X[i][x]   -> at(y,i) = T[y][i]
//   forward  row    pass: Y[y][x] = sum_i M[y][i] T[x][i]   -> at(x,i) = T[x][i]
//   inverse  column pass: M[y][x] = sum_i T[i][y] D[i][x]   -> at(y,i) = T[i][y]
//   inverse  row    pass: R[y][x] = sum_i M[y][i] T[i][x]   -> at(x,i) = T[i][x]
// so the inverse is the forward machinery with T transposed.
template <bool INV, bool CBANK = false>
struct HaweelT {
    static constexpr bool is_static = true;
    static constexpr bool cbank_pairs = CBANK;
    __host__ __device__ static constexpr float at(int a, int i) { return INV ? haweel(i, a) : haweel(a, i); }
    // row-pass output pairing: columns with identical sparsity patterns share an FFMA2
    static constexpr int n_units = INV ? 4 : 5;
    __host__ __device__ static constexpr int ua(int k)
    {
        constexpr int f[5] = {0, 2, 1, 3, 7}, v[4] = {0, 1, 2, 3};
        return INV ? v[k] : f[k];
    }
    __host__ __device__ static constexpr int ub(int k)
    {
        constexpr int f[5] = {4, 6, 5, -1, -1}, v[4] = {7, 6, 5, 4};
        return INV ? v[k] : f[k];
    }
};

template <bool INV>
struct RuntimeT {
    static constexpr bool is_static = false;
    static constexpr bool cbank_pairs = false;
    const DenseT &m;
    __device__ __forceinline__ explicit RuntimeT(const DenseT &mm) : m(mm) {}
    __device__ __forceinline__ float at(int a, int i) const { return INV ? m.tt[a * 8 + i] : m.t[a * 8 + i]; }
    // pair {at(x,i), at(x+1,i)} as one aligned 64-bit constant
    __device__ __forceinline__ float2 at2(int x, int i) const
    {
        const float *base = INV ? m.t : m.tt; // INV: T[i][x],T[i][x+1]; FWD: Tt[i][x],Tt[i][x+1]
        return *reinterpret_cast<const float2 *>(base + i * 8 + x);
    }
    static constexpr int n_units = 4;
    __host__ __device__ static constexpr int ua(int k) { return 2 * k; }
    __host__ __device__ static constexpr int ub(int k) { return 2 * k + 1; }
};

// The five unequal constant pairs of the row passes can live in the constant bank: ptxas then
// fetches them once with LDCU into uniform register pairs (FFMA2 takes UR pairs as operands)
// instead of rebuilding them from immediates with MOVs all over the unrolled code: -100
// instructions per block (1784 -> 1680 in the f32 round trip), same bits.  Measured on one B200
// (profiles/r01_pair_constants.txt): issue-bound kernels gain (u8 direct 70.7 -> 65.4 us, f32
// direct 92.0 -> 88.0); the HBM-bound f32 TMA kernel is 0.9 % slower in a short burst (81.8 ->
// 82.5 us) but 1.3 % faster over 4000 power-capped launches (83.7 -> 82.6 us: fewer instructions,
// less power, same clocks), which is the regime that counts.  All kernels use it; the policy
// stays a template parameter (HaweelT<INV, CBANK>).
static __constant__ float2 c_pairs[6] = {{(float)0.35355339, -(float)0.35355339}, {(float)0.5, -(float)0.5},
                                  {(float)0.4472136, (float)0.2236068}, {(float)0.2236068, -(float)0.4472136},
                                  {(float)0.70710678, -(float)0.70710678}, {1.0f, -1.0f}};
__host__ __device__ constexpr int pair_index(float na, float nb)
{
    return (na == (float)0.35355339) ? 0 : (na == (float)0.5) ? 1 : (na == (float)0.4472136) ? 2
         : (na == (float)0.2236068) ? 3 : 4;
}
template <int I>
__device__ __forceinline__ float2 pair_constant() { return c_pairs[I]; }

// ---------------------------------------------------------------- compile-time retained-coefficient masks
// With the mask known at compile time the dropped coefficients are literal +0.0f: the forward
// chains that feed only dropped positions are never emitted, and the inverse skips every term
// whose coefficient is a known zero.  Skipping is exact for the same reason skipping T's zeros
// is: fma(t, +-0, s) == s bit-for-bit when the running sum s is never -0.0f (it starts at +0.0f),
// and a chain made only of skipped terms yields the +0.0f it started from.
template <uint64_t KEEP>
struct KeepMask {
    static constexpr uint64_t bits = KEEP;
    static constexpr bool all = KEEP == ~0ull;
    __host__ __device__ static constexpr bool kept(int r, int c) { return (KEEP >> (r * 8 + c)) & 1ull; }
    __host__ __device__ static constexpr bool row_any(int r) { return ((KEEP >> (r * 8)) & 0xffull) != 0; }
    __host__ __device__ static constexpr bool col_any(int c) { return ((KEEP >> c) & 0x0101010101010101ull) != 0; }
    __host__ __device__ static constexpr bool pair_any(int r, int j) { return kept(r, 2 * j) || kept(r, 2 * j + 1); }
};
using KeepAll = KeepMask<~0ull>;
// first k positions of the JPEG zig-zag scan (README.md:63 of the reference: 6..10 retained coefficients)
__host__ __device__ constexpr uint64_t zigzag_prefix_mask(int k)
{
    constexpr unsigned char zz[10] = {0, 1, 8, 16, 9, 2, 3, 10, 17, 24};
    uint64_t m = 0;
    for (int i = 0; i < k && i < 10; i++) m |= 1ull << zz[i];
    return m;
}

// ---------------------------------------------------------------- the two passes
// Column pass, in place: for each column pair j, p[y][j] <- chain_i at(y,i) * p[i][j].
// KM (inverse only): input pairs (row i, pair j) outside the mask are known zeros and skipped.
template <class TP, class KM = KeepAll>
__device__ __forceinline__ void col_pass(float2 (&p)[8][4], const TP &tp)
{
    sfor<4>([&](auto j) {
        float2 in[8];
        sfor<8>([&](auto i) { in[IC(i)] = p[IC(i)][IC(j)]; });
        sfor<8>([&](auto y) {
            float2 acc = make_float2(0.0f, 0.0f);
            sfor<8>([&](auto i) {
                if constexpr (TP::is_static) {
                    constexpr float t = TP::at(IC(y), IC(i));
                    if constexpr (t != 0.0f && KM::pair_any(IC(i), IC(j))) acc = ffma2(in[IC(i)], bc(t), acc);
                } else {
                    acc = ffma2(in[IC(i)], bc(tp.at(IC(y), IC(i))), acc);
                }
            });
            p[IC(y)][IC(j)] = acc;
        });
    });
}

// Row pass for one row: o[x] <- chain_i m[i] * at(x,i).
// ZIN::zero(i): m[i] is a known zero (skipped); NEED::need(x): o[x] is used at all (a pair of
// which only one half is needed becomes a scalar chain; unneeded outputs are left untouched).
struct NoZero { __host__ __device__ static constexpr bool zero(int) { return false; } };
struct NeedAll { __host__ __device__ static constexpr bool need(int) { return true; } };
template <class KM> struct ZeroCols { __host__ __device__ static constexpr bool zero(int i) { return !KM::col_any(i); } };
template <class KM, int Y> struct NeedRow { __host__ __device__ static constexpr bool need(int x) { return KM::kept(Y, x); } };

template <class TP, class ZIN, int X>
__device__ __forceinline__ float row_chain_scalar(const float (&m)[8], const TP &tp)
{
    float acc = 0.0f;
    sfor<8>([&](auto i) {
        if constexpr (TP::is_static) {
            constexpr float t = TP::at(X, IC(i));
            if constexpr (t != 0.0f && !ZIN::zero(IC(i))) acc = __fmaf_rn(m[IC(i)], t, acc);
        } else {
            acc = __fmaf_rn(m[IC(i)], tp.at(X, IC(i)), acc);
        }
    });
    return acc;
}

template <class TP, class ZIN = NoZero, class NEED = NeedAll>
__device__ __forceinline__ void row_pass(const float (&m)[8], float (&o)[8], const TP &tp)
{
    sfor<TP::n_units>([&](auto k) {
        constexpr int xa = TP::ua(IC(k)), xb = TP::ub(IC(k));
        constexpr bool need_a = NEED::need(xa), need_b = xb >= 0 && NEED::need(xb);
        if constexpr (need_a && need_b) {
            float2 acc = make_float2(0.0f, 0.0f);
            sfor<8>([&](auto i) {
                if constexpr (TP::is_static) {
                    constexpr float ta = TP::at(xa, IC(i)), tb = TP::at(xb, IC(i));
                    if constexpr ((ta != 0.0f || tb != 0.0f) && !ZIN::zero(IC(i))) {
                        // fma(m,t,c) == fma(-m,-t,c) exactly: normalise the sign of the constant
                        // pair so that only {a,-a},{h,-h},{p,q},{q,-p},{s,-s} ever need registers
                        // (equal halves are broadcast immediates); the sign goes onto m.
                        constexpr bool neg = ta < 0.0f || (ta == 0.0f && tb < 0.0f);
                        constexpr float na = neg ? -ta : ta, nb = neg ? -tb : tb;
                        const float mm = neg ? -m[IC(i)] : m[IC(i)];
                        if constexpr (TP::cbank_pairs && na != nb) acc = ffma2(bc(mm), pair_constant<pair_index(na, nb)>(), acc);
                        else acc = ffma2(bc(mm), make_float2(na, nb), acc);
                    }
                } else {
                    acc = ffma2(bc(m[IC(i)]), tp.at2(xa, IC(i)), acc);
                }
            });
            o[xa] = acc.x;
            o[xb] = acc.y;
        } else if constexpr (need_a) {
            o[xa] = row_chain_scalar<TP, ZIN, xa>(m, tp);
        } else if constexpr (need_b) {
            o[xb] = row_chain_scalar<TP, ZIN, xb>(m, tp);
        }
    });
}

// ---------------------------------------------------------------- quantiser policies
// QImm: the JPEG table as immediates, all coefficients kept (the reference's only
// configuration).  QParam: any table / mask, from the parameter constant bank.
struct QImm {
    static constexpr bool masked = false;
    static constexpr bool fastdiv = true;
    __device__ __forceinline__ float neg_d(int k) const { return -jpeg_q(k); }
    __device__ __forceinline__ float rcp(int k) const { return 1.0f / jpeg_q(k); } // constant-folded, RN
    __device__ __forceinline__ float d(int k) const { return jpeg_q(k); }
    __device__ __forceinline__ uint32_t keep(int) const { return 0xffffffffu; }
};
template <bool MASKED, bool FASTDIV>
struct QParam {
    static constexpr bool masked = MASKED;
    static constexpr bool fastdiv = FASTDIV;
    const QuantTables &q;
    __device__ __forceinline__ explicit QParam(const QuantTables &qq) : q(qq) {}
    __device__ __forceinline__ float neg_d(int k) const { return q.neg_d[k]; }
    __device__ __forceinline__ float rcp(int k) const { return q.rcp[k]; }
    __device__ __forceinline__ float d(int k) const { return q.d[k]; }
    __device__ __forceinline__ uint32_t keep(int k) const { return q.keep[k]; }
};

// round(y / Q[k]) exactly as divide_matrices (utils_kernels.cu:42): IEEE division, then
// round half away from zero (nvcc lowers roundf to copysign(0.5) + add.rz + cvt.rzi).
template <class QP>
__device__ __forceinline__ float quantise(float y, int k, const QP &qp)
{
    float q;
    if constexpr (QP::fastdiv) {
        const float r = qp.rcp(k);
        const float q0 = y * r;
        const float e = __fmaf_rn(q0, qp.neg_d(k), y);
        q = __fmaf_rn(e, r, q0);
    } else {
        q = __fdiv_rn(y, qp.d(k));
    }
    float c = roundf(q);
    if constexpr (QP::masked) c = __uint_as_float(__float_as_uint(c) & qp.keep(k));
    return c;
}

// ---------------------------------------------------------------- whole-block stages
// p holds pixels-128 on entry and the quantised coefficients C on exit.  KM != KeepAll: the mask
// is a compile-time constant, dropped coefficients are +0.0f without being computed (the
// chains that feed only them are dead code) -- same values as computing and masking.
template <class KM = KeepAll, class TF, class QP>
__device__ __forceinline__ void forward_block(float2 (&p)[8][4], const TF &tf, const QP &qp)
{
    col_pass(p, tf);
    sfor<8>([&](auto y) {
        float m[8], o[8];
        sfor<4>([&](auto j) {
            m[2 * IC(j)] = p[IC(y)][IC(j)].x;
            m[2 * IC(j) + 1] = p[IC(y)][IC(j)].y;
        });
        if constexpr (KM::row_any(IC(y))) row_pass<TF, NoZero, NeedRow<KM, IC(y)>>(m, o, tf);
        sfor<4>([&](auto j) {
            if constexpr (KM::kept(IC(y), 2 * IC(j))) p[IC(y)][IC(j)].x = quantise(o[2 * IC(j)], IC(y) * 8 + 2 * IC(j), qp);
            else p[IC(y)][IC(j)].x = 0.0f;
            if constexpr (KM::kept(IC(y), 2 * IC(j) + 1)) p[IC(y)][IC(j)].y = quantise(o[2 * IC(j) + 1], IC(y) * 8 + 2 * IC(j) + 1, qp);
            else p[IC(y)][IC(j)].y = 0.0f;
        });
    });
}

// p holds quantised coefficients C on entry and R = T^T.(C*Q).T on exit (no +128).  KM != KeepAll
// promises that every coefficient outside the mask is +-0 (the caller guarantees it: the fused
// kernels produce them, the inverse-only kernels are not specialised).
template <class KM = KeepAll, class TI, class QP>
__device__ __forceinline__ void inverse_block(float2 (&p)[8][4], const TI &ti, const QP &qp)
{
    sfor<8>([&](auto y) {
        sfor<4>([&](auto j) {
            if constexpr (KM::kept(IC(y), 2 * IC(j))) p[IC(y)][IC(j)].x *= qp.d(IC(y) * 8 + 2 * IC(j)); // multiply_matrices, utils_kernels.cu:55
            if constexpr (KM::kept(IC(y), 2 * IC(j) + 1)) p[IC(y)][IC(j)].y *= qp.d(IC(y) * 8 + 2 * IC(j) + 1);
        });
    });
    col_pass<TI, KM>(p, ti);
    sfor<8>([&](auto y) {
        float m[8], o[8];
        sfor<4>([&](auto j) {
            m[2 * IC(j)] = p[IC(y)][IC(j)].x;
            m[2 * IC(j) + 1] = p[IC(y)][IC(j)].y;
        });
        row_pass<TI, ZeroCols<KM>, NeedAll>(m, o, ti);
        sfor<4>([&](auto j) { p[IC(y)][IC(j)] = make_float2(o[2 * IC(j)], o[2 * IC(j) + 1]); });
    });
}

// ---------------------------------------------------------------- factored inverse (+-1 LSB)
// Haweel's T has symmetric even rows (0,2,4,6) and antisymmetric odd rows (1,3,5,7), so the
// 8-point inverse x[n] = sum_k T[k][n] c[k] splits into x[n] = E[n] + O[n], x[7-n] = E[n] - O[n]:
//     u = a c0 (+bias)   A = u + a c4   B = u - a c4     P = p c2 + q c6   R = q c2 - p c6
//     E0 = A + P   E3 = A - P   E1 = B + R   E2 = B - R
//     x0,x7 = E0 +- h (c1 + c5)   x1,x6 = E1 +- h (c1 - c5)   x2,x5 = E2 -+ s c3   x3,x4 = E3 -+ s c7
// 21 operations instead of the 44 ordered FMAs of the reference chain (cuda_matrix_idct,
// main_newAppr.cu:236-239,246-248).  The sums are re-associated, so the float result differs
// from the chain in the last bits (|diff| <~ 1e-4 at pixel scale): used only where the contract
// is "+-1 LSB" (8-bit pixel output, SURVEY.md section 7.2 "inverse pass has slack"), never for the
// forward transform (quantised coefficients stay bit-exact) and never for f32 pixels.
// Column pass: two adjacent columns per packed instruction, constants broadcast immediates.
// Row pass: the two halves of a packed instruction are the two members of a butterfly, the
// input is a broadcast register and the constant pair {k,-k} comes from the constant bank.
// The +128 of add_matrix_scalar (utils_kernels.cu:29) rides on the DC term of the row pass
// (every output contains u exactly once), so it costs nothing.
template <bool BIAS128, class QP>
__device__ __forceinline__ void inverse_block_fast(float2 (&p)[8][4], const QP &qp)
{
    constexpr float a = (float)0.35355339, h = (float)0.5, pp = (float)0.4472136, q = (float)0.2236068,
                    s = (float)0.70710678;
    sfor<8>([&](auto y) {
        sfor<4>([&](auto j) {
            p[IC(y)][IC(j)].x *= qp.d(IC(y) * 8 + 2 * IC(j)); // multiply_matrices, utils_kernels.cu:55
            p[IC(y)][IC(j)].y *= qp.d(IC(y) * 8 + 2 * IC(j) + 1);
        });
    });
    sfor<4>([&](auto j) {
        const float2 c0 = p[0][IC(j)], c1 = p[1][IC(j)], c2 = p[2][IC(j)], c3 = p[3][IC(j)], c4 = p[4][IC(j)],
                     c5 = p[5][IC(j)], c6 = p[6][IC(j)], c7 = p[7][IC(j)];
        const float2 u = fmul2(c0, bc(a));
        const float2 A = ffma2(c4, bc(a), u), B = ffma2(c4, bc(-a), u);
        const float2 P = ffma2(c6, bc(q), fmul2(c2, bc(pp))), R = ffma2(c6, bc(-pp), fmul2(c2, bc(q)));
        const float2 E0 = fadd2(A, P), E3 = fsub2(A, P), E1 = fadd2(B, R), E2 = fsub2(B, R);
        const float2 sm = fadd2(c1, c5), df = fsub2(c1, c5);
        p[0][IC(j)] = ffma2(sm, bc(h), E0); p[7][IC(j)] = ffma2(sm, bc(-h), E0);
        p[1][IC(j)] = ffma2(df, bc(h), E1); p[6][IC(j)] = ffma2(df, bc(-h), E1);
        p[2][IC(j)] = ffma2(c3, bc(-s), E2); p[5][IC(j)] = ffma2(c3, bc(s), E2);
        p[3][IC(j)] = ffma2(c7, bc(-s), E3); p[4][IC(j)] = ffma2(c7, bc(s), E3);
    });
    sfor<8>([&](auto y) {
        const float m0 = p[IC(y)][0].x, m1 = p[IC(y)][0].y, m2 = p[IC(y)][1].x, m3 = p[IC(y)][1].y,
                    m4 = p[IC(y)][2].x, m5 = p[IC(y)][2].y, m6 = p[IC(y)][3].x, m7 = p[IC(y)][3].y;
        const float u = BIAS128 ? __fmaf_rn(m0, a, 128.0f) : m0 * a;
        const float2 AB = ffma2(bc(m4), pair_constant<0>(), bc(u));                       // {A, B}
        const float2 PR = ffma2(bc(m6), pair_constant<3>(), fmul2(bc(m2), pair_constant<2>())); // {P, R}
        const float2 SD = ffma2(bc(m5), pair_constant<5>(), bc(m1));                      // {c1+c5, c1-c5}
        const float2 E03 = ffma2(bc(PR.x), pair_constant<5>(), bc(AB.x));                 // {E0, E3}
        const float2 E12 = ffma2(bc(PR.y), pair_constant<5>(), bc(AB.y));                 // {E1, E2}
        const float2 x07 = ffma2(bc(SD.x), pair_constant<1>(), bc(E03.x));
        const float2 x16 = ffma2(bc(SD.y), pair_constant<1>(), bc(E12.x));
        const float2 x25 = ffma2(bc(-m3), pair_constant<4>(), bc(E12.y));
        const float2 x34 = ffma2(bc(-m7), pair_constant<4>(), bc(E03.y));
        p[IC(y)][0] = make_float2(x07.x, x16.x); p[IC(y)][1] = make_float2(x25.x, x34.x);
        p[IC(y)][2] = make_float2(x34.y, x25.y); p[IC(y)][3] = make_float2(x16.y, x07.y);
    });
}

// ---------------------------------------------------------------- dense T with even/odd symmetry
// A dense T whose even rows are symmetric (T[k][n] == T[k][7-n]) and whose odd rows are
// antisymmetric (the true DCT-II, and every "exact" matrix the cuBLAS variants of the reference are
// meant for) needs only half the products:
//   forward  y[k] = sum_{n<4} T[k][n] (x[n] +- x[7-n])            8 add/sub + 32 FMA instead of 64 FMA
//   inverse  x[n], x[7-n] = E[n] +- O[n],  E/O[n] = sum_{k even/odd} T[k][n] c[k]   32 FMA + 8 add/sub
// The sums are re-associated with respect to the reference's cuBLAS calls (main_cublass.cu:234-241,
// main_cublass_2.cu:228-235) -- but so is cuBLAS itself with respect to any fixed chain (its
// accumulation order is undocumented; measured 8-54 of 65536 quantised coefficients differ from the
// ascending FMA chain, DESIGN.md section 3), so the criterion for dense T is a mismatch COUNT against the
// live cuBLAS reference, pixels within 1 LSB.  Plans select it automatically when T has the
// structure (b200dct_dense_mode); any other dense T runs the ordered chains.
// Column passes: two adjacent columns per packed instruction, T entries broadcast from the
// parameter bank.  Row passes: the two halves are an (even, odd) pair: {s_n, d_n} = {m[n]+m[7-n],
// m[n]-m[7-n]} feeds {y[2i], y[2i+1]} and {c[2i], c[2i+1]} feeds {E_n, O_n}, so inputs and outputs
// are exactly the natural column pairs p[row][j] -- no re-pairing moves.
template <class QP>
__device__ __forceinline__ void forward_block_sym(float2 (&p)[8][4], const DenseT &m, const QP &qp)
{
    sfor<4>([&](auto j) {
        float2 sd[8]; // [n] = x[n] + x[7-n], [4+n] = x[n] - x[7-n]
        sfor<4>([&](auto n) {
            sd[IC(n)] = fadd2(p[IC(n)][IC(j)], p[7 - IC(n)][IC(j)]);
            sd[4 + IC(n)] = fsub2(p[IC(n)][IC(j)], p[7 - IC(n)][IC(j)]);
        });
        sfor<8>([&](auto k) {
            constexpr int base = (IC(k) & 1) * 4;
            float2 acc = fmul2(sd[base], bc(m.t[IC(k) * 8]));
            sfor<3>([&](auto n) { acc = ffma2(sd[base + 1 + IC(n)], bc(m.t[IC(k) * 8 + 1 + IC(n)]), acc); });
            p[IC(k)][IC(j)] = acc;
        });
    });
    sfor<8>([&](auto y) {
        const float r[8] = {p[IC(y)][0].x, p[IC(y)][0].y, p[IC(y)][1].x, p[IC(y)][1].y,
                            p[IC(y)][2].x, p[IC(y)][2].y, p[IC(y)][3].x, p[IC(y)][3].y};
        float2 sd[4];
        sfor<4>([&](auto n) { sd[IC(n)] = ffma2(bc(r[7 - IC(n)]), pair_constant<5>(), bc(r[IC(n)])); });
        sfor<4>([&](auto i) {
            float2 acc = fmul2(sd[0], m.eo[IC(i) * 4]);
            sfor<3>([&](auto n) { acc = ffma2(sd[1 + IC(n)], m.eo[IC(i) * 4 + 1 + IC(n)], acc); });
            p[IC(y)][IC(i)].x = quantise(acc.x, IC(y) * 8 + 2 * IC(i), qp);
            p[IC(y)][IC(i)].y = quantise(acc.y, IC(y) * 8 + 2 * IC(i) + 1, qp);
        });
    });
}

// C -> pixels WITH the +128 (it rides on the first product of every E_n in the row pass).
template <class QP>
__device__ __forceinline__ void inverse_block_sym(float2 (&p)[8][4], const DenseT &m, const QP &qp)
{
    sfor<8>([&](auto y) {
        sfor<4>([&](auto j) {
            p[IC(y)][IC(j)].x *= qp.d(IC(y) * 8 + 2 * IC(j)); // multiply_matrices, utils_kernels.cu:55
            p[IC(y)][IC(j)].y *= qp.d(IC(y) * 8 + 2 * IC(j) + 1);
        });
    });
    sfor<4>([&](auto j) {
        float2 c[8];
        sfor<8>([&](auto k) { c[IC(k)] = p[IC(k)][IC(j)]; });
        sfor<4>([&](auto n) {
            float2 e = fmul2(c[0], bc(m.t[IC(n)])), o = fmul2(c[1], bc(m.t[8 + IC(n)]));
            sfor<3>([&](auto i) {
                e = ffma2(c[2 + 2 * IC(i)], bc(m.t[(2 + 2 * IC(i)) * 8 + IC(n)]), e);
                o = ffma2(c[3 + 2 * IC(i)], bc(m.t[(3 + 2 * IC(i)) * 8 + IC(n)]), o);
            });
            p[IC(n)][IC(j)] = fadd2(e, o);
            p[7 - IC(n)][IC(j)] = fsub2(e, o);
        });
    });
    sfor<8>([&](auto y) {
        float x[8];
        sfor<4>([&](auto n) {
            float2 eo = ffma2(p[IC(y)][0], m.eo[IC(n)], make_float2(128.0f, 0.0f));
            sfor<3>([&](auto i) { eo = ffma2(p[IC(y)][1 + IC(i)], m.eo[(1 + IC(i)) * 4 + IC(n)], eo); });
            x[IC(n)] = eo.x + eo.y;
            x[7 - IC(n)] = eo.x - eo.y;
        });
        sfor<4>([&](auto j) { p[IC(y)][IC(j)] = make_float2(x[2 * IC(j)], x[2 * IC(j) + 1]); });
    });
}

// ---------------------------------------------------------------- element conversions
// u8 -> (float)b - 128 in two ops: PRMT builds 0x4B0000bb = 2^23 + b, one FADD removes
// 2^23 + 128 (exact).  Equivalent to convertToFloat (utils.cu:13) then sub_matrix_scalar
// (utils_kernels.cu:16).
__device__ __forceinline__ float u8_shifted(uint32_t word, int byte)
{
    const uint32_t bits = __byte_perm(word, 0x4B000000u, 0x7440u | (uint32_t)byte);
    return __uint_as_float(bits) - 8388736.0f;
}
__device__ __forceinline__ float u8_to_float(uint32_t word, int byte)
{
    const uint32_t bits = __byte_perm(word, 0x4B000000u, 0x7440u | (uint32_t)byte);
    return __uint_as_float(bits) - 8388608.0f;
}
// float pixel -> u8 as convertToUnsignedChar (utils.cu:21): clamp to [0,255], then truncate.
// Saturation to [0,255] commutes with truncation toward zero, so "truncate to s32 (saturating,
// NaN -> 0 like fmaxf(NaN, 0)), then saturate to u8" gives the same byte.  Written as
// cvt.rzi.s32.f32 + cvt.pack.sat.u8.s32.b32, which ptxas fuses into ONE two-input
// F2IP.U8.F32.TRUNC per pair of pixels that also merges the previous pair: 2 instructions per 4
// pixels instead of 4 conversions + 3 PRMT (the u8 kernels are issue-bound, DESIGN.md section 4).
__device__ __forceinline__ uint32_t pack4_u8(float a, float b, float c, float d)
{
    const int ia = __float2int_rz(a), ib = __float2int_rz(b), ic = __float2int_rz(c), id = __float2int_rz(d);
    uint32_t hi, w;
    asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, 0;" : "=r"(hi) : "r"(id), "r"(ic));         // bytes {c, d, 0, 0}
    asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(w) : "r"(ib), "r"(ia), "r"(hi)); // bytes {a, b, c, d}
    return w;
}
// integer-valued float coefficient -> saturating int16
__device__ __forceinline__ uint32_t pack2_i16(float a, float b)
{
    short ia, ib;
    asm("cvt.rni.sat.s16.f32 %0, %1;" : "=h"(ia) : "f"(a));
    asm("cvt.rni.sat.s16.f32 %0, %1;" : "=h"(ib) : "f"(b));
    return ((uint32_t)(unsigned short)ia) | ((uint32_t)(unsigned short)ib << 16);
}
// JPEG zig-zag scan (ITU-T T.81 figure 5): position k of the scan -> row*8+col of the block.
__host__ __device__ constexpr int zigzag_pos(int k)
{
    constexpr unsigned char zz[64] = {
        0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5,
        12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21, 28,
        35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51,
        58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
    return zz[k];
}
// the register holding scan position K of a block kept as p[row][column pair]
template <int K>
__device__ __forceinline__ float &zigzag_elem(float2 (&p)[8][4])
{
    constexpr int rc = zigzag_pos(K), r = rc >> 3, c = rc & 7;
    if constexpr (c & 1) return p[r][c >> 1].y;
    else return p[r][c >> 1].x;
}
__device__ __forceinline__ float i16_lo(uint32_t w) { return (float)(short)(w & 0xffffu); }
__device__ __forceinline__ float i16_hi(uint32_t w) { return (float)((int)w >> 16); }

// ---------------------------------------------------------------- host: kernel launch
// One launch of KERNEL with programmatic dependent launch when pdl is set: the kernel may start
// while the previous kernel of the stream drains (every kernel of the library executes
// griddepcontrol.wait before it touches memory its predecessor may write).
// ctas_per_sm != NULL: no launch, only the resident CTAs per SM of KERNEL at this block size and
// dynamic shared memory (cached; a kernel is launched with at most one size besides 0).
template <auto KERNEL, class Params>
inline cudaError_t launch_kernel(const Params &P, dim3 grid, dim3 block, size_t smem, cudaStream_t s, bool pdl,
                                 int *ctas_per_sm = nullptr)
{
    if (ctas_per_sm) {
        static int cached[2] = {-1, -1};
        int &v = cached[smem ? 1 : 0];
        if (v < 0) {
            int n = 0;
            v = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, KERNEL, (int)(block.x * block.y * block.z), smem) == cudaSuccess ? n : 0;
        }
        *ctas_per_sm = v;
        return cudaSuccess;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, KERNEL, P);
}

} // namespace b200dct
