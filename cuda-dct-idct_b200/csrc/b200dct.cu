// b200dct.cu -- host side of the C ABI declared in include/b200dct.h: plans, argument
// checking, kernel-family selection, TMA descriptors, the pipelined host-buffer round
// trip and the device-side MSE/PEEN accumulation.  Plain CUDA C++; no torch, no cuBLAS.
#include "b200dct.h"

#include <cuda.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <mutex>
#include <new>

#include "any_kernels.cuh"
#include "rgb_kernels.cuh"
#include "mma_kernels.cuh"

namespace b200dct {
// one launcher per family and translation unit of kernel instantiations (inst_<family>_<s|d|y><quantiser>.cu, and
// inst_<family>_k.cu for the compile-time masks Q_IMM_K6..K10); ctas_per_sm != NULL: no launch, only the resident-CTA
// count of the kernel the arguments select
#define B200_DECL(tag)                                                                                                  \
    cudaError_t launch_direct_##tag(int qm, int mode, int pix, bool finv, bool metrics, const DirectParams &P, dim3 grid, dim3 block, cudaStream_t s, bool pdl, int *ctas_per_sm); \
    cudaError_t launch_tma_##tag(int qm, int mode, int pix, bool finv, bool metrics, const TmaParams &P, int grid, int block, size_t smem, cudaStream_t s, bool pdl);
B200_DECL(s0) B200_DECL(s1) B200_DECL(s2) B200_DECL(d1) B200_DECL(d2) B200_DECL(y1) B200_DECL(y2) B200_DECL(k)
#undef B200_DECL
cudaError_t launch_any_f32(int tk, int qm, bool finv, const AnyParams &P, dim3 grid, dim3 block, cudaStream_t s, bool pdl); // inst_any_f32.cu
cudaError_t launch_any_u8(int tk, int qm, bool finv, const AnyParams &P, dim3 grid, dim3 block, cudaStream_t s, bool pdl);  // inst_any_u8.cu
cudaError_t launch_mma(bool fastdiv, const MmaParams &P, dim3 grid, dim3 block, cudaStream_t s, bool pdl);                           // inst_mma.cu

struct Unit {
    decltype(&launch_direct_s0) direct;
    decltype(&launch_tma_s0) tma;
};
// the translation unit of (T family, quantiser)
static Unit unit_of(int tk, int q)
{
#define B200_UNIT(tag) Unit{launch_direct_##tag, launch_tma_##tag}
    if (is_kmask(q)) return B200_UNIT(k);
    if (tk == TK_DENSE_SYM) return q == 1 ? B200_UNIT(y1) : B200_UNIT(y2);
    if (tk == TK_HAWEEL) return q == 0 ? B200_UNIT(s0) : q == 1 ? B200_UNIT(s1) : B200_UNIT(s2);
    return q == 1 ? B200_UNIT(d1) : B200_UNIT(d2);
#undef B200_UNIT
}
} // namespace b200dct

using namespace b200dct;

#include "plan_internal.h"

static thread_local int tl_launches = 0;
static thread_local const char *tl_path = "none";
namespace b200dct {
void note_launch(int launches, const char *path)
{
    tl_launches = launches;
    if (path) tl_path = path;
}
} // namespace b200dct

static void plan_refresh(b200dct_plan *pl)
{
    pl->sparse = true;
    pl->q_default = true;
    pl->q_fastdiv = true;
    pl->qc_fastdiv = true;
    for (int k = 0; k < 64; k++) {
        const float h = haweel(k / 8, k % 8);
        if (memcmp(&h, &pl->T[k], 4) != 0 && !(h == 0.0f && pl->T[k] == 0.0f)) pl->sparse = false;
        if (pl->Q[k] != jpeg_q(k)) pl->q_default = false;
        const float d = pl->Q[k];
        if (!(d >= 1.0f && d <= 255.0f && d == floorf(d))) pl->q_fastdiv = false;
        pl->cp.q.d[k] = d;
        pl->cp.q.neg_d[k] = -d;
        pl->cp.q.rcp[k] = 1.0f / d; // IEEE RN on the host
        pl->cp.q.keep[k] = ((pl->mask >> k) & 1) ? 0xffffffffu : 0u;
        const float dc = pl->Qc[k];
        if (!(dc >= 1.0f && dc <= 255.0f && dc == floorf(dc))) pl->qc_fastdiv = false;
        pl->rgb_t[0].rd[k] = make_float2(pl->cp.q.rcp[k], d);
        pl->rgb_t[1].rd[k] = make_float2(1.0f / dc, dc);
        pl->rgb_t[0].keep[k] = pl->rgb_t[1].keep[k] = pl->cp.q.keep[k];
        pl->cp.t.t[k] = pl->T[k];
        pl->cp.t.tt[(k % 8) * 8 + k / 8] = pl->T[k];
    }
    // even rows symmetric, odd rows antisymmetric (exact float comparison): the true DCT-II and
    // every matrix of that family -- evaluated through its even/odd halves unless the plan asks
    // for the ordered chains
    pl->symmetric = true;
    for (int r = 0; r < 8; r++)
        for (int n = 0; n < 4; n++) {
            const float a = pl->T[r * 8 + n], b = pl->T[r * 8 + 7 - n];
            if (!isfinite(a) || ((r & 1) ? (a != -b) : (a != b))) pl->symmetric = false;
        }
    for (int i = 0; i < 4; i++)
        for (int n = 0; n < 4; n++) pl->cp.t.eo[i * 4 + n] = make_float2(pl->T[(2 * i) * 8 + n], pl->T[(2 * i + 1) * 8 + n]);
    pl->tk = pl->sparse ? TK_HAWEEL : ((pl->symmetric && pl->dense != B200DCT_DENSE_CHAIN) ? TK_DENSE_SYM : TK_DENSE);
}

extern "C" int b200dct_plan_create(b200dct_plan **out)
{
    if (!out) return B200DCT_ERR_ARG;
    b200dct_plan *pl = new (std::nothrow) b200dct_plan;
    if (!pl) return B200DCT_ERR_NOMEM;
    for (int k = 0; k < 64; k++) {
        pl->T[k] = haweel(k / 8, k % 8);
        pl->Q[k] = jpeg_q(k);
        pl->Qc[k] = jpeg_q_chroma(k);
    }
    pl->mask = ~(uint64_t)0;
    pl->path = B200DCT_PATH_AUTO;
    // env B200DCT_DENSE=chain|symmetric|auto: default dense-T arithmetic of new plans
    pl->dense = B200DCT_DENSE_AUTO;
    if (const char *e = getenv("B200DCT_DENSE")) {
        if (!strcmp(e, "chain")) pl->dense = B200DCT_DENSE_CHAIN;
        else if (!strcmp(e, "symmetric")) pl->dense = B200DCT_DENSE_SYMMETRIC;
        else if (!strcmp(e, "mma")) pl->dense = B200DCT_DENSE_MMA;
    }
    // env B200DCT_INVERSE=exact|factored|auto: default inverse mode of new plans (a caller that wants
    // the reference's u8 bits everywhere, e.g. through the compat library, sets "exact")
    pl->inverse = B200DCT_INVERSE_AUTO;
    if (const char *e = getenv("B200DCT_INVERSE")) {
        if (!strcmp(e, "exact")) pl->inverse = B200DCT_INVERSE_EXACT;
        else if (!strcmp(e, "factored")) pl->inverse = B200DCT_INVERSE_FACTORED;
    }
    plan_refresh(pl);
    *out = pl;
    return B200DCT_OK;
}

extern "C" void b200dct_plan_destroy(b200dct_plan *pl) { delete pl; }

extern "C" int b200dct_plan_set_quant(b200dct_plan *pl, const float *q)
{
    if (!pl || !q) return B200DCT_ERR_ARG;
    for (int k = 0; k < 64; k++)
        if (!isfinite(q[k]) || q[k] == 0.0f) return B200DCT_ERR_QUANT;
    memcpy(pl->Q, q, sizeof(pl->Q));
    plan_refresh(pl);
    return B200DCT_OK;
}

extern "C" int b200dct_plan_get_quant(const b200dct_plan *pl, float *q)
{
    if (!pl || !q) return B200DCT_ERR_ARG;
    memcpy(q, pl->Q, sizeof(pl->Q));
    return B200DCT_OK;
}

extern "C" int b200dct_plan_set_chroma_quant(b200dct_plan *pl, const float *q)
{
    if (!pl || !q) return B200DCT_ERR_ARG;
    for (int k = 0; k < 64; k++)
        if (!isfinite(q[k]) || q[k] == 0.0f) return B200DCT_ERR_QUANT;
    memcpy(pl->Qc, q, sizeof(pl->Qc));
    plan_refresh(pl);
    return B200DCT_OK;
}

extern "C" int b200dct_plan_get_chroma_quant(const b200dct_plan *pl, float *q)
{
    if (!pl || !q) return B200DCT_ERR_ARG;
    memcpy(q, pl->Qc, sizeof(pl->Qc));
    return B200DCT_OK;
}

extern "C" int b200dct_plan_set_transform(b200dct_plan *pl, const float *t)
{
    if (!pl || !t) return B200DCT_ERR_ARG;
    memcpy(pl->T, t, sizeof(pl->T));
    plan_refresh(pl);
    return B200DCT_OK;
}

extern "C" int b200dct_plan_set_transform_device(b200dct_plan *pl, const void *d_t)
{
    if (!pl || !d_t) return B200DCT_ERR_ARG;
    float t[64];
    cudaError_t e = cudaMemcpy(t, d_t, sizeof(t), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return (int)e;
    return b200dct_plan_set_transform(pl, t);
}

extern "C" int b200dct_plan_set_keep_mask(b200dct_plan *pl, uint64_t mask)
{
    if (!pl) return B200DCT_ERR_ARG;
    pl->mask = mask;
    plan_refresh(pl);
    return B200DCT_OK;
}

extern "C" uint64_t b200dct_zigzag_mask(int k)
{
    static const unsigned char zz[64] = {
        0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5,
        12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21, 28,
        35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51,
        58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
    if (k >= 64) return ~(uint64_t)0;
    uint64_t m = 0;
    for (int i = 0; i < k; i++) m |= (uint64_t)1 << zz[i];
    return m;
}

extern "C" int b200dct_plan_set_path(b200dct_plan *pl, b200dct_path path)
{
    if (!pl || path < B200DCT_PATH_AUTO || path > B200DCT_PATH_TMA) return B200DCT_ERR_ARG;
    pl->path = path;
    return B200DCT_OK;
}

extern "C" int b200dct_plan_set_inverse(b200dct_plan *pl, b200dct_inverse_mode mode)
{
    if (!pl || mode < B200DCT_INVERSE_AUTO || mode > B200DCT_INVERSE_FACTORED) return B200DCT_ERR_ARG;
    pl->inverse = mode;
    return B200DCT_OK;
}

extern "C" int b200dct_plan_set_dense(b200dct_plan *pl, b200dct_dense_mode mode)
{
    if (!pl || mode < B200DCT_DENSE_AUTO || mode > B200DCT_DENSE_MMA) return B200DCT_ERR_ARG;
    pl->dense = mode;
    plan_refresh(pl);
    return B200DCT_OK;
}
// 0 ordered chains, 1 Haweel's sparse kernels, 2 symmetric dense kernels
extern "C" int b200dct_plan_kernel_kind(const b200dct_plan *pl) { return pl ? pl->tk : B200DCT_ERR_ARG; }

// The factored inverse applies to 8-bit pixel output of Haweel's T (contract: +-1 LSB).
static bool use_factored_inverse(const b200dct_plan *pl, int mode, int pix)
{
    return pl->sparse && pix == DT_U8 && mode != MODE_FWD && pl->inverse != B200DCT_INVERSE_EXACT;
}

extern "C" int b200dct_plan_is_sparse(const b200dct_plan *pl) { return pl ? (pl->sparse ? 1 : 0) : B200DCT_ERR_ARG; }

// ------------------------------------------------------------------ device info
struct DevInfo {
    int sms;
    int smem_optin;
    bool ok;
};
static DevInfo dev_info()
{
    static thread_local int cached_dev = -1;
    static thread_local DevInfo info = {0, 0, false};
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess) return DevInfo{0, 0, false};
    if (dev != cached_dev) {
        info.ok = cudaDeviceGetAttribute(&info.sms, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess &&
                  cudaDeviceGetAttribute(&info.smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) == cudaSuccess;
        cached_dev = dev;
    }
    return info;
}

// ------------------------------------------------------------------ TMA descriptors
typedef CUresult (*encode_tiled_fn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                    const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static encode_tiled_fn get_encode()
{
    static encode_tiled_fn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = (encode_tiled_fn)p;
    });
    return fn;
}

static size_t elem_size(int dt) { return dt == DT_F32 ? 4 : ((dt == DT_I16 || dt == DT_I16ZZ) ? 2 : 1); }

// Can this plane be addressed by the tile view of its dtype?
static bool tma_plane_ok(const void *ptr, int dt, size_t pitch, int W)
{
    if (((uintptr_t)ptr & 15) || (pitch & 15)) return false;
    if (dt == DT_I16ZZ) return false; // the block-major zig-zag stream is written by the direct family
    if (dt == DT_F32) return (W % 32) == 0;
    return (((size_t)W * elem_size(dt)) % 16) == 0;
}

static bool make_map(CUtensorMap *map, const void *ptr, int dt, size_t pitch, int H, int W)
{
    encode_tiled_fn enc = get_encode();
    if (!enc) return false;
    CUresult r;
    const CUtensorMapL2promotion promo = CU_TENSOR_MAP_L2_PROMOTION_L2_256B;
    if (dt == DT_F32) {
        // {32 floats, W/32 segments, H rows}; box = 8 rows x 8 segments x 128 B, 128B swizzle
        cuuint64_t dims[3] = {32, (cuuint64_t)(W / 32), (cuuint64_t)H};
        cuuint64_t strides[2] = {128, (cuuint64_t)pitch};
        cuuint32_t box[3] = {32, 8, 8};
        cuuint32_t es[3] = {1, 1, 1};
        r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void *>(ptr), dims, strides, box, es,
                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, promo,
                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    } else {
        cuuint64_t dims[2] = {(cuuint64_t)W, (cuuint64_t)H};
        cuuint64_t strides[1] = {(cuuint64_t)pitch};
        cuuint32_t box[2] = {256, 8};
        cuuint32_t es[2] = {1, 1};
        r = enc(map, dt == DT_U8 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_UINT16, 2,
                const_cast<void *>(ptr), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                CU_TENSOR_MAP_SWIZZLE_NONE, promo, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    }
    return r == CUDA_SUCCESS;
}

// ------------------------------------------------------------------ dispatch
struct Plane {
    const void *ptr;
    int dt;
    size_t pitch;
};

static int check_plane(const Plane &pl, int W, bool pixels)
{
    if (!pl.ptr) return B200DCT_ERR_ARG;
    if (pixels ? (pl.dt != DT_F32 && pl.dt != DT_U8) : (pl.dt != DT_F32 && pl.dt != DT_I16 && pl.dt != DT_I16ZZ)) return B200DCT_ERR_ARG;
    // zig-zag stream: pitch = bytes per block-row = (W/8) blocks x 128 B (= 8 image rows x W x 2 B)
    if (pl.pitch < (size_t)W * elem_size(pl.dt) * (pl.dt == DT_I16ZZ ? 8 : 1)) return B200DCT_ERR_SHAPE;
    const size_t a = pl.dt == DT_U8 ? 8 : 16;
    if (((uintptr_t)pl.ptr % a) || (pl.pitch % a)) return B200DCT_ERR_ALIGN;
    return B200DCT_OK;
}

// Ticket counters of the TMA kernels' dynamic tile scheduler: a per-device ring of
// {next, done} pairs, zero-initialised once; every launch takes the next slot and the kernel
// leaves its slot zeroed again, so launches on different streams never share a live slot
// (that would take SCHED_SLOTS launches in flight at once).
// A launch made under stream capture is replayed many times, possibly while ordinary launches
// walk the ring, so it gets a pair of its own for good from a second pool (CAPTURE_SLOTS per
// device, never recycled): replays of one graph exec are stream-ordered by CUDA and every run
// leaves the pair zeroed.  (Two execs instantiated from the SAME captured graph and replayed
// concurrently would share a pair -- not supported; B200DCT_PATH_DIRECT avoids the counters.)
// Nothing can be allocated during capture, so both pools are created by the first ordinary call.
namespace {
constexpr int SCHED_SLOTS = 4096;
constexpr int CAPTURE_SLOTS = 4096;
struct SchedRing {
    uint32_t *base[64] = {};
    unsigned long long *macc[64] = {}; // one zeroed MACC_WORDS accumulator per slot (metrics kernels)
    unsigned next[64] = {};
    unsigned next_capture[64] = {};
    std::mutex mu;
};
SchedRing g_sched;

uint32_t *sched_slot(bool capturing)
{
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    std::lock_guard<std::mutex> lk(g_sched.mu);
    if (!g_sched.base[dev]) {
        if (capturing) return nullptr;
        uint32_t *p = nullptr;
        const size_t nslots = (size_t)(SCHED_SLOTS + CAPTURE_SLOTS);
        const size_t bytes = nslots * 2 * sizeof(uint32_t) + nslots * MACC_WORDS * sizeof(unsigned long long);
        if (cudaMalloc(&p, bytes) != cudaSuccess) return nullptr;
        if (cudaMemset(p, 0, bytes) != cudaSuccess) { cudaFree(p); return nullptr; }
        g_sched.base[dev] = p;
        g_sched.macc[dev] = reinterpret_cast<unsigned long long *>(p + nslots * 2);
    }
    if (capturing) {
        if (g_sched.next_capture[dev] >= (unsigned)CAPTURE_SLOTS) return nullptr;
        return g_sched.base[dev] + 2 * (SCHED_SLOTS + g_sched.next_capture[dev]++);
    }
    const unsigned s = g_sched.next[dev]++ % SCHED_SLOTS;
    return g_sched.base[dev] + 2 * s;
}
// the integer accumulators that belong to a ticket-counter pair
unsigned long long *sched_macc(const uint32_t *slot)
{
    int dev = -1;
    if (!slot || cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64 || !g_sched.base[dev]) return nullptr;
    return g_sched.macc[dev] + MACC_WORDS * ((slot - g_sched.base[dev]) / 2);
}
// The counters of a fused-metrics launch: those of its scheduler slot, or without one (capture pool used up,
// failed ring allocation) the caller's workspace (METRICS_WORKSPACE_BYTES).  The kernel leaves either zeroed; the
// workspace starts unknown, so a launch on it is preceded by a memset on its stream and takes no part in the early path.
struct MetricsCounters {
    uint32_t *pair; // {next ticket, finished CTAs / warps}
    unsigned long long *macc;
    bool in_workspace;
    // inside the launch's scope, ahead of the kernel
    cudaError_t zero(cudaStream_t s) const { return in_workspace ? cudaMemsetAsync(macc, 0, METRICS_WORKSPACE_BYTES, s) : cudaSuccess; }
};
MetricsCounters metrics_counters(uint32_t *slot, void *workspace)
{
    if (unsigned long long *macc = sched_macc(slot)) return MetricsCounters{slot, macc, false};
    auto *macc = static_cast<unsigned long long *>(workspace);
    return MetricsCounters{reinterpret_cast<uint32_t *>(macc + MACC_WORDS), macc, true};
}
} // namespace

// ---- early tile loads across launch boundaries
// With programmatic dependent launch a kernel's CTAs start while its predecessor drains, but may not
// touch memory before griddepcontrol.wait: at every launch boundary HBM sees a write-only tail followed
// by a read-only ramp (DESIGN.md section 4, "where the last 5 % go").  If nothing the new launch READS is
// written by the launch it can overlap with, its loads need not wait -- only its writes do.  The
// library establishes that by itself, per (device, stream):
//   * the relaxation only ever applies to the immediately preceding kernel of the stream, and only if
//     that kernel triggers launch_dependents -- i.e. one of this library's; what the caller enqueues in
//     between (copies, other kernels) cannot be seen from here and is excluded on the device by the
//     completion counter described further down;
//   * when that predecessor is a persistent TMA-family launch that fills the machine (a CTA on every SM)
//     and both launches take more than half of an SM's shared memory (so they can never share an SM),
//     a successor CTA starts only where a predecessor CTA has EXITED, which it cannot do before
//     having passed its own wait: everything older than the predecessor is complete by the time a
//     successor CTA runs, and only the predecessor's writes matter;
//   * so: predecessor on this stream = such a launch, and [input plane] disjoint from its output /
//     coefficient planes  =>  early tile loads.  Launches that do not qualify as predecessors clear the record.
// Every launch of the library, taking part or not, happens inside a LaunchScope (plan_internal.h), which holds
// g_last_mu across the decision, the launch and the update of the record.
// Not under stream capture.  env B200DCT_EARLY_LOADS=0 disables (A/B).
//
// The direct family (hardware-scheduled 128-thread CTAs, several per SM) has its own version of the argument:
// a dependent launch starts once every CTA of its predecessor has STARTED (executed launch_dependents).
// If the predecessor has more CTAs than the machine can hold at once (grid > resident CTAs per SM x SMs,
// the occupancy of that very kernel), "all started" implies "some exited", and a CTA only exits after its
// griddepcontrol.wait -- so again everything older than the predecessor is complete when a successor CTA
// runs, and only the predecessor's own writes matter.  A direct-family round trip whose input is disjoint
// from them loads AND transforms its blocks before its wait (L2-coherent loads) and only holds back its
// stores: its CTAs work in the slots the predecessor's last wave leaves idle instead of sitting at the wait
// (8192^2 u8: 11 waves of ~5 us, on average half a wave idle per launch boundary).  CTAs beyond one
// machine-full start after the predecessor anyway.
//
// Both arguments are about the library's own kernels; what the CALLER enqueues between two calls is
// invisible to the host side.  A kernel of the caller that writes the next call's input is covered on
// the device: every machine-filling launch feeds a per-(device, stream) completion counter, the host knows
// the value the counter has once the predecessor is complete, and a successor only takes the early path
// when it READS a smaller value -- the predecessor is then provably still running, so nothing enqueued
// after it (which, launched the ordinary way, starts only when the predecessor has completed) can stand
// between the two; otherwise the successor waits first like any dependent launch.  (Not covered: foreign
// kernels themselves launched with programmatic stream serialization between two calls of the library.)
// The device side of the protocol is EarlyPath (dct_kernels.cuh).
namespace b200dct {
struct Range {
    uintptr_t lo = 0, hi = 0; // [lo, hi)
};
struct LastLaunch {
    int dev = -1;
    cudaStream_t stream = nullptr;
    LaunchScope::Family family = LaunchScope::NONE; // of a machine-filling launch that fed the counter, else NONE
    Range w[3];
    bool chain_ok = true; // false once the record has been taken over by another stream (its counter may still be fed)
    unsigned long long expected = 0; // value of the record's completion counter once every recorded launch has completed
};
} // namespace b200dct
namespace {
constexpr int LAST_SLOTS = 16;
LastLaunch g_last[LAST_SLOTS];
unsigned long long *g_chain[64] = {}; // per device: one completion counter per record
std::mutex g_last_mu;
Range plane_range(const Span &sp) { return sp.ptr ? Range{(uintptr_t)sp.ptr, sp.end()} : Range{}; }
bool disjoint(const Range &a, const Range &b) { return a.hi <= b.lo || b.hi <= a.lo || a.lo == a.hi || b.lo == b.hi; }
bool early_loads_enabled()
{
    static const bool v = [] {
        const char *p = getenv("B200DCT_EARLY_LOADS");
        return !(p && atoi(p) == 0);
    }();
    return v;
}
} // namespace
namespace b200dct {
// Before the launch: may a launch of `family` reading `rd` on `s` take the early path, and does it feed the counter?
// Leaves the record cleared; done() fills it in once the kernel is in the stream.
LaunchScope::LaunchScope(cudaStream_t s, Family family, bool usable, unsigned long long ctas, int ctas_per_sm, Span rd, Span w0,
                         Span w1, Span w2)
    : family_(family), w_{w0, w1, w2}
{
    g_last_mu.lock();
    const DevInfo di = dev_info();
    usable = usable && family != NONE && di.ok;
    const unsigned long long machine = (unsigned long long)(ctas_per_sm > 0 ? ctas_per_sm : 0) * (unsigned long long)di.sms;
    // direct style: more CTAs than the machine holds at once; TMA: a CTA on every SM
    const bool fills = usable && machine > 0 && (family == TMA ? ctas >= machine : ctas > machine);
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return;
    LastLaunch *e = nullptr, *freeslot = nullptr;
    for (auto &x : g_last) {
        if (x.dev == dev && x.stream == s) e = &x;
        if (x.dev < 0 && !freeslot) freeslot = &x;
    }
    const bool known = e != nullptr;
    if (!e) {
        if (freeslot) e = freeslot;
        else { // evicting a record is always safe: no early path on it any more
            e = &g_last[((uintptr_t)s >> 4) % LAST_SLOTS];
            e->chain_ok = false;
        }
        e->expected = 0; // a fresh record's counter has never been fed; an evicted one has no counter any more
        e->dev = dev;
        e->stream = s;
        e->family = NONE;
    }
    if (e->chain_ok && !g_chain[dev] && usable) {
        unsigned long long *p = nullptr;
        if (cudaMalloc(&p, LAST_SLOTS * sizeof(unsigned long long)) == cudaSuccess) {
            if (cudaMemset(p, 0, LAST_SLOTS * sizeof(unsigned long long)) == cudaSuccess) g_chain[dev] = p;
            else cudaFree(p);
        }
    }
    rec_ = e;
    unsigned long long *const chain = (e->chain_ok && g_chain[dev]) ? g_chain[dev] + (e - g_last) : nullptr;
    const Range r = usable ? plane_range(rd) : Range{};
    // (TMA family: the successor must not fit beside the predecessor either, i.e. satisfy the condition itself)
    const bool early = known && chain && family != NONE && e->family == family && (family == DIRECT || fills) && r.lo != r.hi &&
                       disjoint(r, e->w[0]) && disjoint(r, e->w[1]) && disjoint(r, e->w[2]) && early_loads_enabled();
    const bool feeds = fills && chain != nullptr;
    e->family = NONE; // until committed
    // the first machine-full of the grid (TMA: the whole grid); the last CTAs of the grid feed (TMA: its last warp out)
    ep_.early = early ? (int)(ctas < machine ? ctas : machine) : 0;
    ep_.chain_feed = feeds ? (family == TMA ? 1 : (int)(ctas < 1024 ? ctas : 1024)) : 0;
    ep_.chain = (feeds || early) ? chain : nullptr;
    ep_.chain_target = e->expected;
}
void LaunchScope::done(bool launched)
{
    if (finished_) return;
    finished_ = true;
    if (launched && rec_) { // this launch as the next one's predecessor
        rec_->family = ep_.chain_feed > 0 ? family_ : NONE;
        for (int i = 0; i < 3; i++) rec_->w[i] = plane_range(w_[i]);
        rec_->expected += (unsigned long long)ep_.chain_feed;
    }
    g_last_mu.unlock();
}
}

// Programmatic dependent launch (default on; env B200DCT_PDL=0 turns it off): consecutive kernels
// of this library in one stream overlap the next kernel's CTA launch and set-up with the previous
// kernel's tail.  Every kernel executes griddepcontrol.wait before its first global-memory access,
// so stream-order data dependencies (forward -> inverse) stay intact.  8192^2 f32 round trip,
// back to back: 83.9 -> 81.8 us (profiles/r01_pdl.txt).
static bool use_pdl()
{
    static const bool v = [] {
        const char *p = getenv("B200DCT_PDL");
        return !(p && atoi(p) == 0);
    }();
    return v;
}
namespace b200dct {
bool use_factored_inverse_u8(const b200dct_plan *pl) { return use_factored_inverse(pl, MODE_RT, DT_U8); }
bool stream_capturing(cudaStream_t s)
{
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    return cudaStreamIsCapturing(s, &cap) == cudaSuccess && cap != cudaStreamCaptureStatusNone;
}
// Under stream capture the attribute would become a programmatic edge of the graph (CUDA >= 12.3):
// no gain on graph replay (82.4 vs 82.2 us at 8192^2 f32, profiles/r01_graph_replay.txt), so captured launches go without.
bool pdl_enabled(bool capturing) { return use_pdl() && !capturing; }
} // namespace b200dct

// AUTO's family choice for a call that moves bytes_per_px (explained where run() makes it)
constexpr unsigned long long TMA_BIG_PIXELS = 28ull << 20, TMA_HUGE_PIXELS = 64ull << 20;
static bool prefers_tma(const b200dct_plan *pl, size_t bytes_per_px, int H, int W)
{
    const unsigned long long px = (unsigned long long)H * (unsigned long long)W;
    return pl->path == B200DCT_PATH_TMA || (bytes_per_px >= 4 && pl->sparse && px >= TMA_BIG_PIXELS) ||
           (bytes_per_px >= 4 && pl->tk == TK_DENSE_SYM && px >= TMA_HUGE_PIXELS);
}

// The kernel variant a plan runs for (mode, pixel dtype): quantiser and the factored inverse.  runtime_mask: the
// kernels take the mask as data only (metrics, any size).
struct Variant {
    int qm;
    bool finv;
};
static Variant variant_of(const b200dct_plan *pl, int mode, int pix, bool runtime_mask)
{
    Variant v;
    if (!pl->q_fastdiv) v.qm = Q_PARAM_DIV;
    else if (pl->sparse && pl->q_default && pl->mask == ~(uint64_t)0) v.qm = Q_IMM;
    else v.qm = Q_PARAM;
    // retained-coefficient round trips (first k = 6..10 zig-zag coefficients of the default
    // tables): kernels with the mask as a compile-time constant
    if (mode == MODE_RT && !runtime_mask && pl->sparse && pl->q_default && pl->q_fastdiv)
        for (int k = 6; k <= 10; k++)
            if (pl->mask == b200dct_zigzag_mask(k)) v.qm = Q_IMM_K6 + (k - 6);
    v.finv = !is_kmask(v.qm) && use_factored_inverse(pl, mode, pix); // compile-time-mask kernels keep the chains
    return v;
}
// the bytes of one plane of a call (the zig-zag stream: H/8 rows of W/8 blocks of 128 bytes)
static Span plane_span(const Plane &p, int H, int W)
{
    if (p.dt == DT_I16ZZ) return Span{p.ptr, p.pitch, (size_t)(W / 8) * 128, H / 8};
    return Span{p.ptr, p.pitch, (size_t)W * elem_size(p.dt), H};
}

// A call of run() whose arguments have passed the checks, and what the family functions share
struct Call {
    const b200dct_plan *pl;
    int mode, pix, coef_dt, H, W;
    Variant v;
    Plane in, out, coef;
    float *shifted;
    cudaStream_t stream;
    bool capturing;
    void *workspace; // fused metrics: the caller's workspace and accumulator (NULL: none)
    double *acc;
    Span rd, w0, w1; // the plane the call reads, the planes it writes
};

// the tensor-core arm of the dense variant (opt-in): f32 fused round trips, optional f32 coefficient plane
static int run_mma(const Call &c)
{
    MmaParams M;
    memset(&M, 0, sizeof(M));
    M.in = (const float *)c.in.ptr; M.in_pitch = c.in.pitch;
    M.out = (float *)const_cast<void *>(c.out.ptr); M.out_pitch = c.out.pitch;
    M.coef = (float *)const_cast<void *>(c.coef.ptr); M.coef_pitch = c.coef.pitch;
    M.bx = c.W / 8; M.by = c.H / 8;
    M.cp = c.pl->cp;
    dim3 grid;
    if (!block_grid(M.by, M.bx, grid)) return B200DCT_ERR_SHAPE;
    return launch_blocks(c.stream, c.capturing, grid, false, Span{}, Span{}, Span{}, Span{}, "mma",
                         [&](const EarlyPath &, bool pdl, int *) { return launch_mma(c.pl->q_fastdiv, M, grid, dim3(32, 4), c.stream, pdl); });
}

// the persistent TMA family; capture_sched: the ticket-counter pair of a captured launch (NULL: none left, or not capturing)
static int run_tma(const Call &c, const DevInfo &di, uint32_t *capture_sched)
{
    const Plane &in = c.in, &out = c.out, &coef = c.coef;
    const int H = c.H, W = c.W;
    TmaParams P;
    memset(&P, 0, sizeof(P));
    if (!make_map(&P.in_map, in.ptr, in.dt, in.pitch, H, W) || !make_map(&P.out_map, out.ptr, out.dt, out.pitch, H, W))
        return B200DCT_ERR_ARG;
    if (coef.ptr && !make_map(&P.coef_map, coef.ptr, coef.dt, coef.pitch, H, W)) return B200DCT_ERR_ARG;
    P.tiles_x = (uint32_t)((W + 255) / 256);
    P.bx = (uint32_t)(W / 8);
    const unsigned long long nt = (unsigned long long)P.tiles_x * (unsigned long long)(H / 8);
    if (nt > 0x7fffffffull) return B200DCT_ERR_SHAPE;
    P.ntiles = (uint32_t)nt;
    P.coef_dt = c.coef_dt;
    P.has_coef = coef.ptr ? 1 : 0;

    // dynamic tickets; a captured launch owns its pair (NULL: no pair left, static split)
    P.sched = c.capturing ? capture_sched : sched_slot(false);
    P.cp = c.pl->cp;
    // tile buffers as large as the largest tile image among the planes of this call
    uint32_t buf = tile_bytes_of(in.dt) > tile_bytes_of(out.dt) ? tile_bytes_of(in.dt) : tile_bytes_of(out.dt);
    if (coef.ptr && tile_bytes_of(coef.dt) > buf) buf = tile_bytes_of(coef.dt);
    P.buf_bytes = buf;
    // warps per CTA: the flavour's CTA size, limited by 227 KiB of shared memory
    int nw = (c.workspace ? TMA_METRICS_THREADS : tma_cta_threads(c.pix, c.pl->tk)) / 32;
    const unsigned nbuf = c.workspace ? 3u : 2u; // metrics: two input buffers per warp
    const int smem_w = (int)((227u * 1024u - 1024u) / (nbuf * buf + 16u));
    if (nw > smem_w) nw = smem_w;
    const size_t smem = (size_t)nw * nbuf * buf + (size_t)nw * 16 + 1024;
    // at most one CTA per SM
    const unsigned long long want = (nt + nw - 1) / nw, sms = (unsigned long long)di.sms;
    const int grid = (int)(want < sms ? want : sms);
    // runs of 2 tiles per ticket while more than two rounds of single tiles remain
    P.run = 2;
    const unsigned long long tail = 2ull * (unsigned long long)grid * nw;
    P.run_tickets = nt > tail ? (uint32_t)((nt - tail) / P.run) : 0u;
    // Metrics: the dynamic scheduler always, on the counters of the slot or of the workspace; the last warp out
    // folds the integer sums into acc -- one launch
    MetricsCounters mc{};
    if (c.workspace) {
        mc = metrics_counters(P.sched, c.workspace);
        P.sched = mc.pair;
        P.macc = mc.macc;
        P.acc = c.acc;
    }
    const bool pdl = pdl_enabled(c.capturing);
    // the argument above needs the predecessor to occupy every SM (grid == SM count) and neither
    // launch to fit beside the other on one SM: both take more than half of its shared memory
    const bool heavy = smem > (size_t)(di.smem_optin / 2) + 1024;
    LaunchScope scope(c.stream, mc.in_workspace ? LaunchScope::NONE : LaunchScope::TMA, pdl && heavy && P.sched != nullptr,
                      (unsigned long long)grid, 1, c.rd, c.w0, c.w1);
    P.ep = scope.early_path();
    const cudaError_t em = mc.zero(c.stream);
    if (em != cudaSuccess) return (int)em;
    const cudaError_t e = unit_of(c.pl->tk, c.v.qm).tma(c.v.qm, c.mode, c.pix, c.v.finv, c.workspace != nullptr, P, grid, nw * 32, smem,
                                                        c.stream, pdl && !mc.in_workspace);
    if (e != cudaSuccess) return (int)e;
    scope.done(true);
    note_launch(1, "tma");
    return B200DCT_OK;
}

// the direct family: hardware-scheduled CTAs, a lane per block
static int run_direct(const Call &c)
{
    DirectParams P;
    memset(&P, 0, sizeof(P));
    P.in = c.in.ptr; P.in_pitch = c.in.pitch;
    P.out = const_cast<void *>(c.out.ptr); P.out_pitch = c.out.pitch;
    P.coef = const_cast<void *>(c.coef.ptr); P.coef_pitch = c.coef.pitch;
    P.shifted = c.shifted; P.shifted_pitch = c.in.pitch;
    P.bx = c.W / 8; P.by = c.H / 8;
    P.coef_dt = c.coef_dt;
    P.zz_smem = (c.coef_dt == DT_I16ZZ && !c.workspace) ? 1 : 0; // the metrics kernels are launched without dynamic smem
    // f32 planes aligned to 32 bytes move with 256-bit accesses
    auto aligned32 = [](const Plane &pl) { return pl.ptr && pl.dt == DT_F32 && !((uintptr_t)pl.ptr & 31) && !(pl.pitch & 31); };
    P.v8 = (aligned32(c.in) ? 1 : 0) | (aligned32(c.out) ? 2 : 0) | (aligned32(c.coef) ? 4 : 0);
    P.cp = c.pl->cp;
    dim3 grid;
    if (!block_grid(P.by, P.bx, grid)) return B200DCT_ERR_SHAPE;
    const bool metrics = c.workspace != nullptr;
    MetricsCounters mc{};
    if (metrics) {
        if (c.mode != MODE_RT || c.in.ptr == c.out.ptr) return B200DCT_ERR_ARG;
        // One launch: integer sums through 64-bit atomics into the accumulator of a ticket-counter pair, the last
        // CTA out folds them into acc (the TMA family's scheme).  Dependent launch and the early path apply on a slot.
        mc = metrics_counters(sched_slot(c.capturing), c.workspace);
        P.macc = mc.macc;
        P.mdone = mc.pair;
        P.acc = c.acc;
    }
    // the early path: fused round trips without a coefficient plane, forward calls without the X-128 write-back,
    // inverse calls whose coefficients are a plane (not the zig-zag stream)
    const bool may_load_early = !c.coef.ptr && !c.shifted && !(c.mode == MODE_INV && c.in.dt == DT_I16ZZ);
    const Span w2 = metrics ? Span{c.acc, 0, 3 * sizeof(double), 1} : Span{c.shifted, c.in.pitch, (size_t)c.W * 4, c.H};
    return launch_blocks(c.stream, c.capturing, grid, true, may_load_early ? c.rd : Span{}, c.w0, c.w1, w2, "direct",
                         [&](const EarlyPath &ep, bool pdl, int *per_sm) {
                             P.ep = ep;
                             return unit_of(c.pl->tk, c.v.qm).direct(c.v.qm, c.mode, c.pix, c.v.finv, metrics, P, grid, dim3(32, 4), c.stream, pdl, per_sm);
                         },
                         mc.in_workspace ? mc.macc : nullptr);
}

static int run(const b200dct_plan *pl, int mode, Plane in, Plane out, Plane coef, float *shifted, int H, int W,
               cudaStream_t stream, void *workspace = nullptr, double *acc = nullptr)
{
    note_launch(0);
    if (!pl) return B200DCT_ERR_ARG;
    if (!whole_blocks(H, W)) return B200DCT_ERR_SHAPE;
    int rc;
    if ((rc = check_plane(in, W, mode != MODE_INV)) != 0) return rc;
    if ((rc = check_plane(out, W, mode != MODE_FWD)) != 0) return rc;
    if (coef.ptr && (rc = check_plane(coef, W, false)) != 0) return rc;
    if (mode == MODE_RT && in.dt != out.dt) return B200DCT_ERR_ARG;
    if (shifted && (in.dt != DT_F32 || mode != MODE_FWD)) return B200DCT_ERR_ARG;

    const DevInfo di = dev_info();
    if (!di.ok) return B200DCT_ERR_NODEVICE;

    const int pix = (mode == MODE_INV) ? out.dt : in.dt;
    const int coef_dt = (mode == MODE_FWD) ? out.dt : (mode == MODE_INV ? in.dt : (coef.ptr ? coef.dt : DT_F32));
    // the metrics kernels take runtime masks
    const Call c{pl, mode, pix, coef_dt, H, W, variant_of(pl, mode, pix, workspace != nullptr), in, out, coef, shifted, stream,
                 stream_capturing(stream), workspace, acc, plane_span(in, H, W), plane_span(out, H, W), plane_span(coef, H, W)};

    // AUTO: the TMA family wins where the call is HBM-bound (>= 4 bytes moved per pixel: any
    // f32/i16 plane); all-u8 round trips move 2 B/px, are instruction-issue bound, and run faster
    // on the direct family (64.5 vs 67 us at 8192^2 with the TMA family at 16 warps, round 1).
    const size_t bytes_per_px = elem_size(in.dt) + elem_size(out.dt) + (coef.ptr ? elem_size(coef.dt) : 0);
    // Dense T (32 FMA/px instead of 22) is issue bound as well: direct 92.5 us vs TMA 112 us.
    // Below ~28 Mpixel the persistent kernel's fixed costs (descriptor fetch, barrier set-up,
    // one CTA per SM) lose to the direct family (C-loop timings with dependent launch,
    // profiles/r01_small_sizes.txt): 256^2 3.4 vs 6.7 us, 2048^2 7.9 vs 9.7, 4096^2 22.9 vs 24.6,
    // 5120^2 34.9 vs 35.0, 6144^2 48.9 vs 48.0, 8192^2 83.8 vs 81.8.
    // (TMA_BIG_PIXELS = 28 Mpixel)
    // Symmetric dense T (16+16 FMA/px).  Before early tile loads the direct family won up to 12288^2
    // (84.6 vs 88.0 us at 8192^2, 187.7 vs 189.0 at 12288^2) and the persistent TMA kernel beyond
    // (16384^2: 321.9 vs 333.9 us); with early loads across launch boundaries the TMA family wins from
    // 8192^2 on: 80.2 vs 84.7 us, 16384^2 314.7 vs 330.9 us (profiles/r02_dense_paths.txt).  Ordered-chain
    // dense kernels stay on the direct family.
    // (TMA_HUGE_PIXELS = 64 Mpixel)
    const bool prefer_tma = prefers_tma(pl, bytes_per_px, H, W);
    // fused metrics on the TMA family: f32 round trips of Haweel's T (the input tile is compared where it
    // already is, in shared memory); everything else takes the direct family's metrics kernels
    const bool metrics_tma_ok = !workspace || (mode == MODE_RT && in.dt == DT_F32 && pl->tk == TK_HAWEEL && in.ptr != out.ptr);
    const bool tma_possible = pl->path != B200DCT_PATH_DIRECT && prefer_tma && !shifted && metrics_tma_ok && get_encode() != nullptr &&
                              tma_plane_ok(in.ptr, in.dt, in.pitch, W) && tma_plane_ok(out.ptr, out.dt, out.pitch, W) &&
                              (!coef.ptr || tma_plane_ok(coef.ptr, coef.dt, coef.pitch, W));
    // Under stream capture the launch takes a ticket-counter pair of its own (see SchedRing); when
    // none is left (or the pools do not exist yet) AUTO falls back to the hardware-scheduled
    // direct family (86.9 us at 8192^2), which beats the TMA family's static split (99.8 us).
    uint32_t *capture_sched = nullptr;
    if (c.capturing && tma_possible) capture_sched = sched_slot(true);
    const bool use_tma = tma_possible && !(c.capturing && !capture_sched && pl->path == B200DCT_PATH_AUTO);
    if (pl->path == B200DCT_PATH_TMA && !use_tma) return B200DCT_ERR_ALIGN;
    if (pl->dense == B200DCT_DENSE_MMA && !pl->sparse && mode == MODE_RT && in.dt == DT_F32 && !workspace && !shifted &&
        (!coef.ptr || coef.dt == DT_F32))
        return run_mma(c);
    if (use_tma) return run_tma(c, di, capture_sched);
    return run_direct(c);
}

extern "C" int b200dct_forward(const b200dct_plan *plan, const void *img, b200dct_dtype img_dt, size_t img_pitch,
                               void *coef, b200dct_dtype coef_dt, size_t coef_pitch, void *shifted_or_null, int H,
                               int W, void *stream)
{
    return run(plan, MODE_FWD, Plane{img, (int)img_dt, img_pitch}, Plane{coef, (int)coef_dt, coef_pitch},
               Plane{nullptr, DT_F32, 0}, (float *)shifted_or_null, H, W, (cudaStream_t)stream);
}

extern "C" int b200dct_inverse(const b200dct_plan *plan, const void *coef, b200dct_dtype coef_dt, size_t coef_pitch,
                               void *img, b200dct_dtype img_dt, size_t img_pitch, int H, int W, void *stream)
{
    return run(plan, MODE_INV, Plane{coef, (int)coef_dt, coef_pitch}, Plane{img, (int)img_dt, img_pitch},
               Plane{nullptr, DT_F32, 0}, nullptr, H, W, (cudaStream_t)stream);
}

extern "C" int b200dct_roundtrip(const b200dct_plan *plan, const void *img, b200dct_dtype in_dt, size_t in_pitch,
                                 void *out, b200dct_dtype out_dt, size_t out_pitch, void *coef_or_null,
                                 b200dct_dtype coef_dt, size_t coef_pitch, int H, int W, void *stream)
{
    return run(plan, MODE_RT, Plane{img, (int)in_dt, in_pitch}, Plane{out, (int)out_dt, out_pitch},
               Plane{coef_or_null, (int)coef_dt, coef_pitch}, nullptr, H, W, (cudaStream_t)stream);
}

// ------------------------------------------------------------------ batches of separately allocated images
// One launch per DIRECT_BATCH_MAX images (the third grid dimension walks the images, their plane
// pointers travel in the kernel parameters: no device-side table, no copy, legal under stream
// capture); consecutive launches of a longer batch overlap through programmatic dependent launch.
// The direct family: hardware-scheduled CTAs need no per-image tensor maps, and it is the family
// the small images a batch is made of run on anyway.
extern "C" int b200dct_roundtrip_batch(const b200dct_plan *plan, int n_images, const void *const *imgs, void *const *outs,
                                       b200dct_dtype dt, size_t in_pitch, size_t out_pitch, int H, int W, void *stream)
{
    note_launch(0);
    if (!plan || n_images < 0 || (n_images > 0 && (!imgs || !outs))) return B200DCT_ERR_ARG;
    if (dt != B200DCT_F32 && dt != B200DCT_U8) return B200DCT_ERR_ARG;
    if (!whole_blocks(H, W)) return B200DCT_ERR_SHAPE;
    for (int i = 0; i < n_images; i++) {
        int rc;
        if ((rc = check_plane(Plane{imgs[i], (int)dt, in_pitch}, W, true)) != 0) return rc;
        if ((rc = check_plane(Plane{outs[i], (int)dt, out_pitch}, W, true)) != 0) return rc;
    }
    if (n_images == 0) return B200DCT_OK;
    const DevInfo di = dev_info();
    if (!di.ok) return B200DCT_ERR_NODEVICE;
    cudaStream_t s = (cudaStream_t)stream;
    // Images large enough for the persistent TMA kernels to win (f32 from 28 Mpixel, see run()) go through
    // the single-image path one by one: consecutive launches overlap (dependent launch, early tile loads),
    // 79.5 against 86 us per 8192^2 f32 image on the direct family.
    if (plan->path != B200DCT_PATH_DIRECT && prefers_tma(plan, 2 * elem_size((int)dt), H, W)) {
        int launches = 0;
        const char *path = "none";
        for (int i = 0; i < n_images; i++) {
            const int rc = run(plan, MODE_RT, Plane{imgs[i], (int)dt, in_pitch}, Plane{outs[i], (int)dt, out_pitch},
                               Plane{nullptr, DT_F32, 0}, nullptr, H, W, s);
            if (rc != B200DCT_OK) return rc;
            launches += tl_launches;
            path = tl_path;
        }
        note_launch(launches, path);
        return B200DCT_OK;
    }
    const Variant v = variant_of(plan, MODE_RT, (int)dt, false);
    const bool pdl = pdl_enabled(stream_capturing(s));
    DirectParams P;
    memset(&P, 0, sizeof(P));
    P.in_pitch = in_pitch; P.out_pitch = out_pitch;
    P.bx = W / 8; P.by = H / 8;
    P.coef_dt = DT_F32;
    P.cp = plan->cp;
    bool v8 = dt == B200DCT_F32 && !(in_pitch & 31) && !(out_pitch & 31);
    for (int i = 0; v8 && i < n_images; i++) v8 = !((uintptr_t)imgs[i] & 31) && !((uintptr_t)outs[i] & 31);
    P.v8 = v8 ? 3 : 0;
    dim3 grid;
    if (!block_grid(P.by, P.bx, grid)) return B200DCT_ERR_SHAPE;
    LaunchScope order(s);
    int launches = 0;
    for (int first = 0; first < n_images; first += DIRECT_BATCH_MAX) {
        const int n = n_images - first < DIRECT_BATCH_MAX ? n_images - first : DIRECT_BATCH_MAX;
        P.nimg = n;
        for (int i = 0; i < n; i++) {
            P.img_in[i] = imgs[first + i];
            P.img_out[i] = outs[first + i];
        }
        P.in = P.img_in[0]; P.out = P.img_out[0];
        grid.z = (unsigned)n;
        const cudaError_t e = unit_of(plan->tk, v.qm).direct(v.qm, MODE_RT, (int)dt, v.finv, false, P, grid, dim3(32, 4), s, pdl, nullptr);
        if (e != cudaSuccess) return (int)e;
        launches++;
    }
    note_launch(launches, "direct");
    return B200DCT_OK;
}

// ------------------------------------------------------------------ any size / any alignment
extern "C" int b200dct_roundtrip_any(const b200dct_plan *plan, const void *img, b200dct_dtype dt, size_t in_pitch,
                                     void *out, size_t out_pitch, int H, int W, void *stream)
{
    note_launch(0);
    if (!plan || !img || !out || H <= 0 || W <= 0) return B200DCT_ERR_ARG;
    if (dt != B200DCT_F32 && dt != B200DCT_U8) return B200DCT_ERR_ARG;
    const size_t es = elem_size((int)dt);
    if (in_pitch < (size_t)W * es || out_pitch < (size_t)W * es) return B200DCT_ERR_SHAPE;
    if (((uintptr_t)img % es) || ((uintptr_t)out % es) || (in_pitch % es) || (out_pitch % es)) return B200DCT_ERR_ALIGN;
    const size_t al = dt == B200DCT_U8 ? 8 : 16;
    const bool fast = whole_blocks(H, W) && !((uintptr_t)img % al) && !((uintptr_t)out % al) && !(in_pitch % al) &&
                      !(out_pitch % al);
    if (fast) return b200dct_roundtrip(plan, img, dt, in_pitch, out, dt, out_pitch, nullptr, B200DCT_F32, 0, H, W, stream);
    // everything else: one pass of the edge-replicating scalar-access kernel, no scratch image
    const DevInfo di = dev_info();
    if (!di.ok) return B200DCT_ERR_NODEVICE;
    cudaStream_t s = (cudaStream_t)stream;
    AnyParams P;
    memset(&P, 0, sizeof(P));
    P.in = img; P.in_pitch = in_pitch;
    P.out = out; P.out_pitch = out_pitch;
    P.H = H; P.W = W;
    P.cp = plan->cp;
    const Variant v = variant_of(plan, MODE_RT, (int)dt, true); // finv only for 8-bit pixels
    dim3 grid;
    if (!block_grid((H + 7) / 8, (W + 7) / 8, grid)) return B200DCT_ERR_SHAPE;
    const auto launch_any = dt == B200DCT_F32 ? launch_any_f32 : launch_any_u8;
    return launch_blocks(s, stream_capturing(s), grid, false, Span{}, Span{}, Span{}, Span{}, "any",
                         [&](const EarlyPath &, bool pdl, int *) { return launch_any(plan->tk, v.qm, v.finv, P, grid, dim3(32, 4), s, pdl); });
}

extern "C" size_t b200dct_metrics_workspace_bytes(int H, int W)
{
    return H > 0 && W > 0 ? METRICS_WORKSPACE_BYTES : 0;
}

extern "C" int b200dct_roundtrip_metrics(const b200dct_plan *plan, const void *img, b200dct_dtype in_dt, size_t in_pitch,
                                         void *out, b200dct_dtype out_dt, size_t out_pitch, void *coef_or_null,
                                         b200dct_dtype coef_dt, size_t coef_pitch, int H, int W, double *d_acc3,
                                         void *workspace, size_t workspace_bytes, void *stream)
{
    if (!d_acc3 || !workspace || workspace_bytes < b200dct_metrics_workspace_bytes(H, W) || ((uintptr_t)workspace & 7))
        return B200DCT_ERR_ARG;
    return run(plan, MODE_RT, Plane{img, (int)in_dt, in_pitch}, Plane{out, (int)out_dt, out_pitch},
               Plane{coef_or_null, (int)coef_dt, coef_pitch}, nullptr, H, W, (cudaStream_t)stream, workspace,
               d_acc3);
}

// Average device time of `iters` back-to-back identical calls, measured with CUDA events on
// `stream` from C (no interpreter between launches).  which: 0 roundtrip(a -> b [,c = coef]),
// 1 forward(a -> b), 2 inverse(a -> b), 3 forward(a -> c) then inverse(c -> b).
extern "C" int b200dct_time_calls(const b200dct_plan *plan, int which, const void *a, b200dct_dtype a_dt, size_t a_pitch,
                                  void *b, b200dct_dtype b_dt, size_t b_pitch, void *c, b200dct_dtype c_dt,
                                  size_t c_pitch, int H, int W, int iters, float *ms_per_iter, void *stream)
{
    if (!ms_per_iter || iters < 1) return B200DCT_ERR_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    cudaEvent_t e0, e1;
    if (cudaEventCreate(&e0) != cudaSuccess || cudaEventCreate(&e1) != cudaSuccess) return B200DCT_ERR_NODEVICE;
    int rc = B200DCT_OK, launches = 0;
    auto once = [&]() -> int {
        switch (which) {
        case 0: return b200dct_roundtrip(plan, a, a_dt, a_pitch, b, b_dt, b_pitch, c, c_dt, c_pitch, H, W, stream);
        case 1: return b200dct_forward(plan, a, a_dt, a_pitch, b, b_dt, b_pitch, nullptr, H, W, stream);
        case 2: return b200dct_inverse(plan, a, a_dt, a_pitch, b, b_dt, b_pitch, H, W, stream);
        case 3: {
            int r = b200dct_forward(plan, a, a_dt, a_pitch, c, c_dt, c_pitch, nullptr, H, W, stream);
            return r ? r : b200dct_inverse(plan, c, c_dt, c_pitch, b, b_dt, b_pitch, H, W, stream);
        }
        default: return B200DCT_ERR_ARG;
        }
    };
    for (int i = 0; i < 3 && rc == B200DCT_OK; i++) rc = once(); // warm-up
    if (rc == B200DCT_OK) {
        cudaEventRecord(e0, s);
        for (int i = 0; i < iters && rc == B200DCT_OK; i++) {
            rc = once();
            launches += tl_launches * (which == 3 ? 2 : 1);
        }
        cudaEventRecord(e1, s);
        cudaError_t e = cudaEventSynchronize(e1);
        if (rc == B200DCT_OK && e != cudaSuccess) rc = (int)e;
        float ms = 0.0f;
        if (rc == B200DCT_OK && cudaEventElapsedTime(&ms, e0, e1) == cudaSuccess) *ms_per_iter = ms / (float)iters;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    note_launch(launches);
    return rc;
}

// ------------------------------------------------------------------ metrics
template <class T>
__global__ void k_metrics(const T *__restrict__ a, const T *__restrict__ b, size_t pitch_elems, int H, int W, double *acc)
{
    double se = 0.0, en = 0.0;
    for (long long y = blockIdx.x; y < H; y += gridDim.x) {
        const T *ra = a + (size_t)y * pitch_elems, *rb = b + (size_t)y * pitch_elems;
        for (int x = threadIdx.x; x < W; x += blockDim.x) {
            const double va = (double)ra[x], d = va - (double)rb[x];
            se += d * d;
            en += va * va;
        }
    }
    for (int o = 16; o > 0; o >>= 1) {
        se += __shfl_xor_sync(0xffffffffu, se, o);
        en += __shfl_xor_sync(0xffffffffu, en, o);
    }
    __shared__ double s_se[32], s_en[32];
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) { s_se[w] = se; s_en[w] = en; }
    __syncthreads();
    if (w == 0) {
        se = l < (blockDim.x >> 5) ? s_se[l] : 0.0;
        en = l < (blockDim.x >> 5) ? s_en[l] : 0.0;
        for (int o = 16; o > 0; o >>= 1) {
            se += __shfl_xor_sync(0xffffffffu, se, o);
            en += __shfl_xor_sync(0xffffffffu, en, o);
        }
        if (l == 0) { atomicAdd(&acc[0], se); atomicAdd(&acc[1], en); }
    }
}

extern "C" int b200dct_metrics_accumulate(const void *ref_img, const void *test_img, b200dct_dtype dt, size_t pitch,
                                          int H, int W, double *d_acc, void *stream)
{
    note_launch(0);
    if (!ref_img || !test_img || !d_acc || H <= 0 || W <= 0) return B200DCT_ERR_ARG;
    const DevInfo di = dev_info();
    if (!di.ok) return B200DCT_ERR_NODEVICE;
    int grid = di.sms * 8 < H ? di.sms * 8 : H;
    if (dt == B200DCT_F32)
        k_metrics<float><<<grid, 256, 0, (cudaStream_t)stream>>>((const float *)ref_img, (const float *)test_img, pitch / 4, H, W, d_acc);
    else if (dt == B200DCT_U8)
        k_metrics<unsigned char><<<grid, 256, 0, (cudaStream_t)stream>>>((const unsigned char *)ref_img, (const unsigned char *)test_img, pitch, H, W, d_acc);
    else
        return B200DCT_ERR_ARG;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return (int)e;
    note_launch(1);
    return B200DCT_OK;
}

// ------------------------------------------------------------------ self-test: constant division
// Sweeps every float bit pattern x in [first, first+count) and compares the kernels'
// three-FMA division by d against __fdiv_rn (the reference's div.rn.f32).  out[0] counts
// finite x with |x| >= 2^-120 whose QUOTIENT bits differ (below that the residual
// underflows and the last bit of a subnormal-range quotient may differ; it rounds to the
// same +-0), out[1] those whose quantised value roundf(quotient) differs (the only thing
// the transform consumes).  x = -0.0f is skipped: the fast path returns +0 for it, and the
// transform can never produce it (an fma chain that starts from +0 never yields -0).
__global__ void k_selftest_div(float d, unsigned long long first, unsigned long long count, unsigned long long *out)
{
    const float nd = -d, r = 1.0f / d;
    unsigned long long bad_q = 0, bad_c = 0;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < count;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        const float x = __uint_as_float((unsigned)(first + i));
        if (!isfinite(x) || (unsigned)(first + i) == 0x80000000u) continue;
        const float q0 = x * r;
        const float e = __fmaf_rn(q0, nd, x);
        const float q = __fmaf_rn(e, r, q0);
        const float ref = __fdiv_rn(x, d);
        if (__float_as_uint(q) != __float_as_uint(ref) && fabsf(x) >= 0x1p-120f) bad_q++;
        if (__float_as_uint(roundf(q)) != __float_as_uint(roundf(ref))) bad_c++;
    }
    if (bad_q) atomicAdd(&out[0], bad_q);
    if (bad_c) atomicAdd(&out[1], bad_c);
}

extern "C" int b200dct_selftest_division(float d, unsigned long long first, unsigned long long count,
                                         unsigned long long *d_out2, void *stream)
{
    if (!d_out2 || !(d != 0.0f)) return B200DCT_ERR_ARG;
    const DevInfo di = dev_info();
    if (!di.ok) return B200DCT_ERR_NODEVICE;
    k_selftest_div<<<di.sms * 16, 256, 0, (cudaStream_t)stream>>>(d, first, count, d_out2);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? B200DCT_OK : (int)e;
}

// Launches made under stream capture take a ticket-counter pair for good (CUDA offers no hook to
// return it when the graph is destroyed): a long-lived process that keeps re-capturing can ask how
// many are left; once they are gone captured AUTO launches take the direct family (b200dct_last_path
// says "direct"), they never fail.
extern "C" int b200dct_capture_slots_left(void)
{
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return B200DCT_ERR_NODEVICE;
    std::lock_guard<std::mutex> lk(g_sched.mu);
    return CAPTURE_SLOTS - (int)g_sched.next_capture[dev];
}

extern "C" int b200dct_last_launch_count(void) { return tl_launches; }
extern "C" const char *b200dct_last_path(void) { return tl_path; }

extern "C" const char *b200dct_error_string(int err)
{
    switch (err) {
    case B200DCT_OK: return "ok";
    case B200DCT_ERR_ARG: return "bad argument (NULL pointer, dtype not valid for that plane, or mixed pixel dtypes)";
    case B200DCT_ERR_SHAPE: return "H and W must be positive multiples of 8 and pitch >= row bytes";
    case B200DCT_ERR_ALIGN: return "pointer/pitch not aligned (16 B for f32/i16 planes, 8 B for u8), or TMA path forced on an unsuitable layout";
    case B200DCT_ERR_NODEVICE: return "no usable CUDA device (this library has no CPU fallback)";
    case B200DCT_ERR_QUANT: return "quantisation entries must be finite and non-zero";
    case B200DCT_ERR_NOMEM: return "out of memory";
    default: return err > 0 ? cudaGetErrorString((cudaError_t)err) : "unknown error";
    }
}

extern "C" int b200dct_version(void) { return B200DCT_VERSION; }
