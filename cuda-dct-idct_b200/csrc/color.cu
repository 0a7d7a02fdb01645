// color.cu -- host side of the colour entry points (b200dct_roundtrip_rgb, b200dct_forward_rgb,
// b200dct_inverse_rgb) and of the coded-size / compression-factor kernel (b200dct_zigzag_coded_bits).  See rgb_kernels.cuh for the arithmetic.
#include <cuda_runtime.h>
#include <string.h>

#include "plan_internal.h"

using namespace b200dct;

// ctas_per_sm != NULL: no launch, only the occupancy of kernel k (`occupancy`: the caller's cache of it)
static cudaError_t launch_rgb_kernel(void (*k)(RgbParams), int &occupancy, const RgbParams &P, dim3 grid, cudaStream_t s,
                                     bool pdl, int *ctas_per_sm)
{
    if (ctas_per_sm) {
        if (occupancy < 0) {
            int n = 0;
            occupancy = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k, 128, 0) == cudaSuccess ? n : 0;
        }
        *ctas_per_sm = occupancy;
        return cudaSuccess;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = dim3(32, 4);
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, k, P);
}
using RgbLauncher = cudaError_t (*)(const RgbParams &, dim3, cudaStream_t, bool, int *);
template <int QK, bool FINV, bool ZZ>
static cudaError_t launch_rgb3(const RgbParams &P, dim3 grid, cudaStream_t s, bool pdl, int *ctas_per_sm)
{
    static int occupancy = -1;
    return launch_rgb_kernel(k_rgb<QK, FINV, ZZ>, occupancy, P, grid, s, pdl, ctas_per_sm);
}
template <int QK>
static cudaError_t launch_rgb_forward(const RgbParams &P, dim3 grid, cudaStream_t s, bool pdl, int *ctas_per_sm)
{
    static int occupancy = -1;
    return launch_rgb_kernel(k_rgb_forward<QK>, occupancy, P, grid, s, pdl, ctas_per_sm);
}
template <bool FINV>
static cudaError_t launch_rgb_inverse(const RgbParams &P, dim3 grid, cudaStream_t s, bool pdl, int *ctas_per_sm)
{
    static int occupancy = -1;
    return launch_rgb_kernel(k_rgb_inverse<FINV>, occupancy, P, grid, s, pdl, ctas_per_sm);
}

// The argument rules of the colour entry points and the parameters their kernels share.  rgb_in / rgb_out: the pixel
// planes the call has (NULL where it has none), interleaved RGB with 8-byte aligned rows; zz: the three streams
// (NULL: none), 16-byte aligned, planes >= (H/8)*(W/8)*128 bytes apart.
static int rgb_params(const b200dct_plan *plan, const void *rgb_in, size_t in_pitch, void *rgb_out, size_t out_pitch,
                      void *zz, size_t zz_plane_bytes, int H, int W, RgbParams &P, dim3 &grid)
{
    if (H <= 0 || W <= 0 || (H % 8) || (W % 8)) return B200DCT_ERR_SHAPE;
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
    for (int k = 0; k < 64; k++) {
        P.t[0].rd[k] = make_float2(plan->cp.q.rcp[k], plan->cp.q.d[k]);
        P.t[0].keep[k] = plan->cp.q.keep[k];
        P.t[1].rd[k] = make_float2(plan->qc.rcp[k], plan->qc.d[k]);
        P.t[1].keep[k] = plan->qc.keep[k];
    }
    grid = dim3((unsigned)((P.by + 3) / 4), (unsigned)((P.bx + 31) / 32));
    if (grid.y > 65535u) return B200DCT_ERR_SHAPE;
    return B200DCT_OK;
}
static Span rgb_span(const void *p, size_t pitch, int H, int W) { return Span{p, pitch, (size_t)W * 3, H}; }
static Span zz_span(const void *zz, size_t plane_bytes, int H, int W) { return Span{zz, plane_bytes, (size_t)(H / 8) * (size_t)(W / 8) * 128, 3}; }
// quantiser variant of the forward transform: 0 all coefficients kept, exact fast division; 1 mask + exact fast
// division; 2 mask + __fdiv_rn
static int rgb_qk(const b200dct_plan *plan)
{
    return (!plan->q_fastdiv || !plan->qc_fastdiv) ? 2 : (plan->mask == ~(uint64_t)0 ? 0 : 1);
}
// One launch of a colour kernel.  Early path across launch boundaries (b200dct.cu, "early loads"): a pass whose
// input `rd` is not written by the library's previous machine-filling launch on this stream reads and computes
// before it waits (rd.ptr NULL: never); w0 / w1 are what the launch writes.
static int run_rgb(RgbLauncher launch, RgbParams &P, dim3 grid, cudaStream_t s, Span rd, Span w0, Span w1)
{
    const bool pdl = pdl_enabled(s);
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    const bool capturing = cudaStreamIsCapturing(s, &cap) == cudaSuccess && cap != cudaStreamCaptureStatusNone;
    int per_sm = 0;
    if (pdl && !capturing) launch(P, grid, s, pdl, &per_sm);
    cudaError_t e;
    {
        EarlyScope scope(s, pdl && !capturing, (unsigned long long)grid.x * grid.y, per_sm, rd, w0, w1);
        P.early = scope.params().early;
        P.chain_feed = scope.params().chain_feed;
        P.chain = scope.params().chain;
        P.chain_target = scope.params().chain_target;
        e = launch(P, grid, s, pdl, nullptr);
        scope.done(e == cudaSuccess);
    }
    if (e != cudaSuccess) return (int)e;
    note_launch(1, "rgb");
    return B200DCT_OK;
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
        {{launch_rgb3<0, false, false>, launch_rgb3<0, false, true>}, {launch_rgb3<0, true, false>, launch_rgb3<0, true, true>}},
        {{launch_rgb3<1, false, false>, launch_rgb3<1, false, true>}, {launch_rgb3<1, true, false>, launch_rgb3<1, true, true>}},
        {{launch_rgb3<2, false, false>, launch_rgb3<2, false, true>}, {launch_rgb3<2, true, false>, launch_rgb3<2, true, true>}}};
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
    static const RgbLauncher launchers[3] = {launch_rgb_forward<0>, launch_rgb_forward<1>, launch_rgb_forward<2>};
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
    static const RgbLauncher launchers[2] = {launch_rgb_inverse<false>, launch_rgb_inverse<true>};
    return run_rgb(launchers[use_factored_inverse_u8(plan)], P, grid, (cudaStream_t)stream, zz_span(zz3, zz_plane_bytes, H, W),
                   rgb_span(out, out_pitch, H, W), Span{nullptr, 0, 0, 0});
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
    if (H <= 0 || W <= 0 || (H % 8) || (W % 8) || pitch < (size_t)(W / 8) * 128) return B200DCT_ERR_SHAPE;
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
