// plan_internal.h -- the plan object behind the opaque b200dct_plan handle (host TUs only).
#pragma once
#include <initializer_list>

#include "b200dct.h"
#include "any_kernels.cuh"
#include "rgb_kernels.cuh"

struct b200dct_plan {
    float T[64];
    float Q[64];
    float Qc[64];    // chrominance table of the colour entry point (default: ITU-T T.81 Annex K.2)
    uint64_t mask;
    bool sparse;     // T is bit-identical to Haweel's matrix
    bool q_default;  // Q is the JPEG luminance table
    bool q_fastdiv;  // every divisor is in the exhaustively proven set (integers 1..255)
    int path;        // b200dct_path
    int inverse;     // b200dct_inverse_mode
    int dense;       // b200dct_dense_mode
    bool symmetric;  // dense T whose even rows are symmetric and odd rows antisymmetric
    int tk;          // TK_HAWEEL / TK_DENSE_SYM / TK_DENSE: the kernels this plan runs
    b200dct::CommonParams cp; // device-ready tables
    b200dct::PlaneTables rgb_t[2]; // the colour kernels' tables: [0] luminance (Q), [1] chrominance (Qc), same mask
    bool qc_fastdiv; // as q_fastdiv, for Qc
};


namespace b200dct {
struct Span {
    const void *ptr; size_t pitch, row_bytes; int rows; // rows of row_bytes, pitch bytes apart
    uintptr_t end() const { return (uintptr_t)ptr + (size_t)(rows - 1) * pitch + row_bytes; } // past the last byte
};
// one span from the lowest start to the highest end of `spans` (conservative where they lie apart)
inline Span span_hull(std::initializer_list<Span> spans)
{
    uintptr_t lo = ~(uintptr_t)0, hi = 0;
    for (const Span &x : spans) {
        lo = (uintptr_t)x.ptr < lo ? (uintptr_t)x.ptr : lo;
        hi = x.end() > hi ? x.end() : hi;
    }
    return Span{(const void *)lo, hi - lo, hi - lo, 1};
}
struct LastLaunch; // the (device, stream) record of b200dct.cu
// Every launch of a library kernel happens inside one of these (see "early loads" in b200dct.cu).  The scope
// holds the launch-order lock from its decision until done() or its end, so that the per-(device, stream)
// record of the last launch follows stream order even when several host threads launch on one stream.
class LaunchScope {
public:
    // DIRECT: hardware-scheduled 128-thread CTAs (direct family, colour), ctas_per_sm = the kernel's occupancy;
    // TMA: persistent kernel, ctas_per_sm = 1.  usable: programmatic dependent launch is on for this launch, the
    // stream is not capturing, and (TMA) the kernel feeds the completion counter and no two of its CTAs fit on
    // one SM.  rd: the plane the launch reads (ptr NULL: never early); w0..w2: the planes it writes.
    enum Family { NONE, DIRECT, TMA };
    LaunchScope(cudaStream_t s, Family family, bool usable, unsigned long long ctas, int ctas_per_sm, Span rd, Span w0,
                Span w1 = Span{}, Span w2 = Span{});
    // a launch (or several) that does not take part in the early path: the record is left cleared
    explicit LaunchScope(cudaStream_t s) : LaunchScope(s, NONE, false, 0, 0, Span{}, Span{}) {}
    ~LaunchScope() { done(false); }
    LaunchScope(const LaunchScope &) = delete;
    LaunchScope &operator=(const LaunchScope &) = delete;
    // the decision, for the kernel's parameters
    const EarlyPath &early_path() const { return ep_; }
    // launched: the scope's kernels are in the stream and the record describes them from now on; releases the lock
    void done(bool launched);
private:
    Family family_;
    EarlyPath ep_{};
    LastLaunch *rec_ = nullptr;
    Span w_[3];
    bool finished_ = false;
};
// b200dct_last_launch_count / b200dct_last_path of this thread (path NULL: left as it is)
void note_launch(int launches, const char *path = nullptr);
bool use_factored_inverse_u8(const b200dct_plan *pl);
bool stream_capturing(cudaStream_t s);
bool pdl_enabled(bool capturing); // programmatic dependent launch for a launch (never on a capturing stream)

// The caller's metrics workspace: {u64 macc[MACC_WORDS]; u32 pair[2]} (see MetricsCounters in b200dct.cu)
constexpr size_t METRICS_WORKSPACE_BYTES = MACC_WORDS * sizeof(unsigned long long) + 2 * sizeof(uint32_t);

// H and W positive multiples of m: whole 8 x 8 blocks, or (m = 16) whole 4:2:0 MCUs
inline bool whole_blocks(int H, int W, int m = 8) { return H > 0 && W > 0 && !(H % m) && !(W % m); }

// Grid of a kernel of 32 x 4-thread CTAs over by x bx blocks: a lane per block, a warp per 32 blocks of a block-row,
// a CTA per 4 block-rows.  false: more than 65535 CTAs across a row (B200DCT_ERR_SHAPE).
inline bool block_grid(int by, int bx, dim3 &grid)
{
    grid = dim3((unsigned)((by + 3) / 4), (unsigned)((bx + 31) / 32));
    return grid.y <= 65535u;
}

// One launch of a kernel of hardware-scheduled 32 x 4-thread CTAs (direct family, any size, tensor-core arm, colour) in
// the library's launch order: dependent launch unless the stream is capturing; with `early`, a part in the early path
// (LaunchScope::DIRECT at the occupancy of the very kernel) reading rd (ptr NULL: never early) and writing w0 .. w2.  This
// thread's last launch is `path`.  launch(ep, pdl, ctas_per_sm) launches with the decision ep (the kernels without an
// early path ignore it), or with ctas_per_sm != NULL only reports the kernel's resident CTAs per SM.
// workspace: the metrics workspace the kernel counts in (NULL: none), zeroed on the stream inside the scope ahead of the
// kernel; its contents are unknown before that, so such a launch takes no part in the early path and has no dependent launch.
template <class Launch>
int launch_blocks(cudaStream_t s, bool capturing, dim3 grid, bool early, Span rd, Span w0, Span w1, Span w2, const char *path,
                  Launch &&launch, void *workspace = nullptr)
{
    const bool pdl = pdl_enabled(capturing) && !workspace;
    const bool part = early && !workspace;
    const bool usable = part && pdl;
    int per_sm = 0;
    if (usable) launch(EarlyPath{}, pdl, &per_sm);
    LaunchScope scope(s, part ? LaunchScope::DIRECT : LaunchScope::NONE, usable, (unsigned long long)grid.x * grid.y, per_sm, rd,
                      w0, w1, w2);
    if (workspace) {
        const cudaError_t e = cudaMemsetAsync(workspace, 0, METRICS_WORKSPACE_BYTES, s);
        if (e != cudaSuccess) return (int)e;
    }
    const cudaError_t e = launch(scope.early_path(), pdl, nullptr);
    if (e != cudaSuccess) return (int)e;
    scope.done(true);
    note_launch(1, path);
    return B200DCT_OK;
}
}
