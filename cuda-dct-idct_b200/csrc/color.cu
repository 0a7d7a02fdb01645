// color.cu -- host side of the colour entry points (b200dct_roundtrip_rgb, b200dct_forward_rgb,
// b200dct_inverse_rgb, and with 4:2:0 chroma b200dct_forward_rgb420, b200dct_inverse_rgb420) and of the coded-size /
// compression-factor kernel (b200dct_zigzag_coded_bits).  See rgb_kernels.cuh and rgb420_kernels.cuh for the arithmetic.
#include <cuda_runtime.h>
#include <string.h>

#include "plan_internal.h"
#include "rgb420_kernels.cuh"

using namespace b200dct;

// launch_kernel (dct_core.cuh) of one colour kernel
using RgbLauncher = cudaError_t (*)(const RgbParams &, dim3, dim3, size_t, cudaStream_t, bool, int *);

// The argument rules of the colour entry points and the parameters their kernels share.  rgb_in / rgb_out: the pixel
// planes the call has (NULL where it has none), interleaved RGB with 8-byte aligned rows; zz: the three streams
// (NULL: none), 16-byte aligned, planes >= (H/8)*(W/8)*128 bytes apart.
static int rgb_params(const b200dct_plan *plan, const void *rgb_in, size_t in_pitch, void *rgb_out, size_t out_pitch,
                      void *zz, size_t zz_plane_bytes, int H, int W, RgbParams &P, dim3 &grid)
{
    if (!whole_blocks(H, W)) return B200DCT_ERR_SHAPE;
    if ((rgb_in && in_pitch < (size_t)W * 3) || (rgb_out && out_pitch < (size_t)W * 3)) return B200DCT_ERR_SHAPE;
    if (((uintptr_t)rgb_in & 7) || ((uintptr_t)rgb_out & 7) || (in_pitch & 7) || (out_pitch & 7)) return B200DCT_ERR_ALIGN;
    if (!plan->sparse) return B200DCT_ERR_ARG; // the colour path is built for Haweel's T (the reference's HpApprDCT)
    const size_t zz_bytes = (size_t)(H / 8) * (size_t)(W / 8) * 128;
    if (zz && (((uintptr_t)zz & 15) || (zz_plane_bytes & 15) || zz_plane_bytes < zz_bytes)) return B200DCT_ERR_ALIGN;
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess) return B200DCT_ERR_NODEVICE;

    memset(&P, 0, sizeof(P));
    P.in = rgb_in; P.in_pitch = in_pitch;
    P.out = rgb_out; P.out_pitch = out_pitch;
    P.zz = zz; P.zz_plane = zz_plane_bytes; P.zz_pitch = (size_t)(W / 8) * 128;
    P.bx = W / 8; P.by = H / 8;
    memcpy(P.t, plan->rgb_t, sizeof(P.t));
    return block_grid(P.by, P.bx, grid) ? B200DCT_OK : B200DCT_ERR_SHAPE;
}
static Span rgb_span(const void *p, size_t pitch, int H, int W) { return Span{p, pitch, (size_t)W * 3, H}; }
static Span zz_span(const void *zz, size_t plane_bytes, int H, int W) { return Span{zz, plane_bytes, (size_t)(H / 8) * (size_t)(W / 8) * 128, 3}; }
// quantiser variant of the forward transform: 0 all coefficients kept, exact fast division; 1 mask + exact fast
// division; 2 mask + __fdiv_rn
static int rgb_qk(const b200dct_plan *plan)
{
    return (!plan->q_fastdiv || !plan->qc_fastdiv) ? 2 : (plan->mask == ~(uint64_t)0 ? 0 : 1);
}
// One launch of a colour kernel, in the early path across launch boundaries (b200dct.cu, "early loads"): a pass whose
// input `rd` is not written by the library's previous machine-filling launch on this stream reads and computes
// before it waits (rd.ptr NULL: never); w0 .. w2 are what the launch writes.
template <class Params> // RgbParams, Rgb420Params
static int run_rgb(cudaError_t (*launch)(const Params &, dim3, dim3, size_t, cudaStream_t, bool, int *), Params &P, dim3 grid,
                   cudaStream_t s, Span rd, Span w0, Span w1, Span w2 = Span{})
{
    return launch_blocks(s, stream_capturing(s), grid, true, rd, w0, w1, w2, "rgb", [&](const EarlyPath &ep, bool pdl, int *per_sm) {
        P.ep = ep;
        return launch(P, grid, dim3(32, 4), 0, s, pdl, per_sm);
    });
}

extern "C" int b200dct_roundtrip_rgb(const b200dct_plan *plan, const void *rgb, size_t in_pitch, void *out,
                                     size_t out_pitch, void *zz3_or_null, size_t zz_plane_bytes, int H, int W,
                                     void *stream)
{
    note_launch(0, "none");
    if (!plan || !rgb || !out) return B200DCT_ERR_ARG;
    RgbParams P;
    dim3 grid;
    const int rc = rgb_params(plan, rgb, in_pitch, out, out_pitch, zz3_or_null, zz_plane_bytes, H, W, P, grid);
    if (rc != B200DCT_OK) return rc;
    static const RgbLauncher launchers[3][2][2] = {
        {{launch_kernel<k_rgb<0, false, false>>, launch_kernel<k_rgb<0, false, true>>},
         {launch_kernel<k_rgb<0, true, false>>, launch_kernel<k_rgb<0, true, true>>}},
        {{launch_kernel<k_rgb<1, false, false>>, launch_kernel<k_rgb<1, false, true>>},
         {launch_kernel<k_rgb<1, true, false>>, launch_kernel<k_rgb<1, true, true>>}},
        {{launch_kernel<k_rgb<2, false, false>>, launch_kernel<k_rgb<2, false, true>>},
         {launch_kernel<k_rgb<2, true, false>>, launch_kernel<k_rgb<2, true, true>>}}};
    // with streams every CTA writes mid-kernel, so that kernel never takes the early path
    return run_rgb(launchers[rgb_qk(plan)][use_factored_inverse_u8(plan)][zz3_or_null != nullptr], P, grid, (cudaStream_t)stream,
                   rgb_span(zz3_or_null ? nullptr : rgb, in_pitch, H, W), rgb_span(out, out_pitch, H, W),
                   zz_span(zz3_or_null, zz_plane_bytes, H, W));
}

extern "C" int b200dct_forward_rgb(const b200dct_plan *plan, const void *rgb, size_t in_pitch, void *zz3,
                                   size_t zz_plane_bytes, int H, int W, void *stream)
{
    note_launch(0, "none");
    if (!plan || !rgb || !zz3) return B200DCT_ERR_ARG;
    RgbParams P;
    dim3 grid;
    const int rc = rgb_params(plan, rgb, in_pitch, nullptr, 0, zz3, zz_plane_bytes, H, W, P, grid);
    if (rc != B200DCT_OK) return rc;
    static const RgbLauncher launchers[3] = {launch_kernel<k_rgb_forward<0>>, launch_kernel<k_rgb_forward<1>>,
                                             launch_kernel<k_rgb_forward<2>>};
    return run_rgb(launchers[rgb_qk(plan)], P, grid, (cudaStream_t)stream, rgb_span(rgb, in_pitch, H, W),
                   zz_span(zz3, zz_plane_bytes, H, W), Span{nullptr, 0, 0, 0});
}

extern "C" int b200dct_inverse_rgb(const b200dct_plan *plan, const void *zz3, size_t zz_plane_bytes, void *out,
                                   size_t out_pitch, int H, int W, void *stream)
{
    note_launch(0, "none");
    if (!plan || !zz3 || !out) return B200DCT_ERR_ARG;
    RgbParams P;
    dim3 grid;
    const int rc = rgb_params(plan, nullptr, 0, out, out_pitch, const_cast<void *>(zz3), zz_plane_bytes, H, W, P, grid);
    if (rc != B200DCT_OK) return rc;
    static const RgbLauncher launchers[2] = {launch_kernel<k_rgb_inverse<false>>, launch_kernel<k_rgb_inverse<true>>};
    return run_rgb(launchers[use_factored_inverse_u8(plan)], P, grid, (cudaStream_t)stream, zz_span(zz3, zz_plane_bytes, H, W),
                   rgb_span(out, out_pitch, H, W), Span{nullptr, 0, 0, 0});
}

// ------------------------------------------------------------------ 4:2:0 chroma (rgb420_kernels.cuh)
using Rgb420Launcher = cudaError_t (*)(const Rgb420Params &, dim3, dim3, size_t, cudaStream_t, bool, int *);

// The argument rules of the 4:2:0 entry points: those of the 4:4:4 calls, H and W multiples of 16, and three
// tightly packed streams, each 16-byte aligned.
// grid: the forward kernel's (16 x 2 MCUs per CTA)
static int rgb420_params(const b200dct_plan *plan, const void *rgb_in, size_t in_pitch, void *rgb_out, size_t out_pitch,
                         const void *zy, const void *zcb, const void *zcr, int H, int W, Rgb420Params &P, dim3 &grid)
{
    if (!whole_blocks(H, W, 16)) return B200DCT_ERR_SHAPE;
    if ((rgb_in && in_pitch < (size_t)W * 3) || (rgb_out && out_pitch < (size_t)W * 3)) return B200DCT_ERR_SHAPE;
    if (((uintptr_t)rgb_in & 7) || ((uintptr_t)rgb_out & 7) || (in_pitch & 7) || (out_pitch & 7)) return B200DCT_ERR_ALIGN;
    if (((uintptr_t)zy & 15) || ((uintptr_t)zcb & 15) || ((uintptr_t)zcr & 15)) return B200DCT_ERR_ALIGN;
    if (!plan->sparse) return B200DCT_ERR_ARG; // Haweel's T only, as the 4:4:4 calls
    if (!block_grid(H / 8, W / 8, grid)) return B200DCT_ERR_SHAPE;
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess) return B200DCT_ERR_NODEVICE;

    memset(&P, 0, sizeof(P));
    P.in = rgb_in; P.in_pitch = in_pitch;
    P.out = rgb_out; P.out_pitch = out_pitch;
    P.zz[0] = const_cast<void *>(zy); P.zz[1] = const_cast<void *>(zcb); P.zz[2] = const_cast<void *>(zcr);
    P.zz_pitch[0] = (size_t)(W / 8) * 128; P.zz_pitch[1] = (size_t)(W / 16) * 128;
    P.mx = W / 16; P.my = H / 16;
    memcpy(P.t, plan->rgb_t, sizeof(P.t));
    return B200DCT_OK;
}
static Span y_span(const void *zz, int H, int W) { return Span{zz, (size_t)(W / 8) * 128, (size_t)(W / 8) * 128, H / 8}; }
static Span c_span(const void *zz, int H, int W) { return Span{zz, (size_t)(W / 16) * 128, (size_t)(W / 16) * 128, H / 16}; }
extern "C" int b200dct_forward_rgb420(const b200dct_plan *plan, const void *rgb, size_t in_pitch, void *zz_y, void *zz_cb,
                                      void *zz_cr, int H, int W, void *stream)
{
    note_launch(0, "none");
    if (!plan || !rgb || !zz_y || !zz_cb || !zz_cr) return B200DCT_ERR_ARG;
    Rgb420Params P;
    dim3 grid;
    const int rc = rgb420_params(plan, rgb, in_pitch, nullptr, 0, zz_y, zz_cb, zz_cr, H, W, P, grid);
    if (rc != B200DCT_OK) return rc;
    static const Rgb420Launcher launchers[3] = {launch_kernel<k_rgb420_forward<0>>, launch_kernel<k_rgb420_forward<1>>,
                                                launch_kernel<k_rgb420_forward<2>>};
    return run_rgb(launchers[rgb_qk(plan)], P, grid, (cudaStream_t)stream, rgb_span(rgb, in_pitch, H, W), y_span(zz_y, H, W),
                      c_span(zz_cb, H, W), c_span(zz_cr, H, W));
}

extern "C" int b200dct_inverse_rgb420(const b200dct_plan *plan, const void *zz_y, const void *zz_cb, const void *zz_cr,
                                      void *out, size_t out_pitch, int H, int W, void *stream)
{
    note_launch(0, "none");
    if (!plan || !zz_y || !zz_cb || !zz_cr || !out) return B200DCT_ERR_ARG;
    Rgb420Params P;
    dim3 grid;
    const int rc = rgb420_params(plan, nullptr, 0, out, out_pitch, zz_y, zz_cb, zz_cr, H, W, P, grid);
    if (rc != B200DCT_OK) return rc;
    static const Rgb420Launcher launchers[2] = {launch_kernel<k_rgb420_inverse<false>>, launch_kernel<k_rgb420_inverse<true>>};
    grid = dim3((unsigned)((P.my + R420_MY - 1) / R420_MY), (unsigned)((P.mx + R420_MX - 1) / R420_MX));
    // the early path's read span: one range over the three streams
    return run_rgb(launchers[use_factored_inverse_u8(plan)], P, grid, (cudaStream_t)stream,
                   span_hull({y_span(zz_y, H, W), c_span(zz_cb, H, W), c_span(zz_cr, H, W)}), rgb_span(out, out_pitch, H, W), Span{}, Span{});
}

// ------------------------------------------------------------------ coded size of a coefficient stream
// Baseline-JPEG (ITU-T T.81 sequential Huffman, Annex K.3 tables = what libjpeg writes) size in bits
// of the entropy-coded scan of ONE plane's zig-zag stream: per block the DC difference to the
// previous block in raster order, (run, size) codes for the AC coefficients, ZRL for runs of 16
// zeros, EOB.  This is the denominator of the compression factor the reference's README reports
// (README.md:62-69) -- CF = 8*H*W / bits.  One thread per block; code lengths from two 256-byte
// tables in shared memory.
namespace {
struct HuffLengths {
    unsigned char dc[2][16];
    unsigned char ac[2][256];
};
HuffLengths make_lengths()
{
    static const unsigned char dc_bits[2][16] = {{0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0},
                                                 {0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0}};
    static const unsigned char ac_bits[2][16] = {{0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 0x7d},
                                                 {0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 0x77}};
    // HUFFVAL of the two AC tables: symbols in order of increasing code length
    static const unsigned char ac_vals[2][162] = {
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
    HuffLengths h;
    memset(&h, 0, sizeof(h));
    for (int t = 0; t < 2; t++) {
        int k = 0;
        for (int l = 1; l <= 16; l++)
            for (int i = 0; i < dc_bits[t][l - 1]; i++) h.dc[t][k++] = (unsigned char)l; // HUFFVAL of the DC tables is 0..11
        k = 0;
        for (int l = 1; l <= 16; l++)
            for (int i = 0; i < ac_bits[t][l - 1]; i++) h.ac[t][ac_vals[t][k++]] = (unsigned char)l;
    }
    return h;
}
const HuffLengths &lengths()
{
    static const HuffLengths h = make_lengths();
    return h;
}
struct CodedParams {
    const void *zz;
    size_t pitch; // bytes per block-row of the stream
    int bx, by;
    int table;
    unsigned long long *bits;
    HuffLengths h;
};
__device__ __forceinline__ int bit_size(int v) { return 32 - __clz(v < 0 ? -v : v); } // T.81 F.1.2.1 SSSS
} // namespace

static __global__ void __launch_bounds__(256) k_coded_bits(const __grid_constant__ CodedParams P)
{
    __shared__ unsigned char acl[256];
    __shared__ unsigned char dcl[16];
    __shared__ unsigned long long cta_bits;
    acl[threadIdx.x] = P.h.ac[P.table][threadIdx.x];
    if (threadIdx.x < 16) dcl[threadIdx.x] = P.h.dc[P.table][threadIdx.x];
    if (threadIdx.x == 0) cta_bits = 0;
    __syncthreads();
    const long long nblk = (long long)P.bx * P.by;
    unsigned bits = 0;
    bool out_of_range = false;
    for (long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x; b < nblk; b += (long long)gridDim.x * blockDim.x) {
        const long long r = b / P.bx;
        const int c = (int)(b - r * P.bx);
        const uint4 *blk = reinterpret_cast<const uint4 *>((const char *)P.zz + (size_t)r * P.pitch + (size_t)c * 128);
        // DC of the previous block in raster order (0 for the first block of the plane)
        int prev = 0;
        if (b > 0) {
            const long long pr = c ? r : r - 1;
            const int pc = c ? c - 1 : P.bx - 1;
            prev = *reinterpret_cast<const short *>((const char *)P.zz + (size_t)pr * P.pitch + (size_t)pc * 128);
        }
        int run = 0;
        // baseline JPEG codes DC-difference categories 0..11 and AC categories 1..10 only: a symbol outside them has no
        // code, counts 0 bits and sets the flag (bit 63 of *P.bits); no table is indexed with it
#pragma unroll
        for (int g = 0; g < 8; g++) {
            const uint4 w = __ldg(blk + g);
            const uint32_t ws[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
            for (int k = 0; k < 8; k++) {
                const int v = (int)(short)(ws[k >> 1] >> (16 * (k & 1)));
                if (g == 0 && k == 0) {
                    const int s = bit_size(v - prev);
                    if (s <= 11) bits += dcl[s] + s;
                    else out_of_range = true;
                } else if (v == 0) {
                    run++;
                } else {
                    while (run > 15) { bits += acl[0xf0]; run -= 16; }
                    const int s = bit_size(v);
                    if (s <= 10) bits += acl[(run << 4) | s] + s;
                    else out_of_range = true;
                    run = 0;
                }
            }
        }
        if (run) bits += acl[0x00];
    }
    unsigned long long v = bits;
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(&cta_bits, v);
    __syncthreads();
    if (threadIdx.x == 0 && cta_bits) atomicAdd(P.bits, cta_bits); // integer sums: order does not matter
    if (__any_sync(0xffffffffu, out_of_range) && (threadIdx.x & 31) == 0) atomicOr(P.bits, B200DCT_CODED_OUT_OF_RANGE);
}

extern "C" int b200dct_zigzag_coded_bits(const void *zz, size_t pitch, int H, int W, int table,
                                         unsigned long long *d_bits, void *stream)
{
    note_launch(0, "none");
    if (!zz || !d_bits || (table != 0 && table != 1)) return B200DCT_ERR_ARG;
    if (!whole_blocks(H, W) || pitch < (size_t)(W / 8) * 128) return B200DCT_ERR_SHAPE;
    if (((uintptr_t)zz & 15) || (pitch & 15) || ((uintptr_t)d_bits & 7)) return B200DCT_ERR_ALIGN;
    int dev = -1, sms = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
        return B200DCT_ERR_NODEVICE;
    CodedParams P;
    P.zz = zz; P.pitch = pitch; P.bx = W / 8; P.by = H / 8; P.table = table; P.bits = d_bits;
    P.h = lengths();
    const long long nblk = (long long)P.bx * P.by;
    long long grid = (nblk + 255) / 256;
    if (grid > (long long)sms * 8) grid = (long long)sms * 8;
    k_coded_bits<<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(P);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return (int)e;
    note_launch(1, "coded_bits");
    return B200DCT_OK;
}
