// plan_internal.h -- the plan object behind the opaque b200dct_plan handle (host TUs only).
#pragma once
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
    b200dct::QuantTables qc; // device-ready chrominance tables (same mask)
    bool qc_default, qc_fastdiv;
};


namespace b200dct {
struct Span { const void *ptr; size_t pitch, row_bytes; int rows; }; // rows of row_bytes, pitch bytes apart
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
    // the decision in the kernel's parameters
    template <class DirectStyleParams> // DirectParams, RgbParams
    void apply(DirectStyleParams &P) const
    {
        P.early = early_;
        P.chain_feed = chain_feed_;
        P.chain = chain_;
        P.chain_target = chain_target_;
    }
    void apply(TmaParams &P) const
    {
        P.early_loads = early_;
        P.chain_feed = chain_feed_;
        P.chain = chain_;
        P.chain_target = chain_target_;
    }
    // launched: the scope's kernels are in the stream and the record describes them from now on; releases the lock
    void done(bool launched);
private:
    Family family_;
    int early_ = 0;                       // leading CTAs that may load before griddepcontrol.wait (TMA: 1 = early tile loads)
    int chain_feed_ = 0;                  // what the kernel adds to the completion counter in total
    unsigned long long *chain_ = nullptr; // completion counter of the (device, stream) record
    unsigned long long chain_target_ = 0; // its value once the predecessor is complete
    void *rec_ = nullptr;                 // the (device, stream) record of b200dct.cu
    Span w_[3];
    bool finished_ = false;
};
void note_launch(int launches, const char *path); // b200dct_last_launch_count / b200dct_last_path of this thread
bool use_factored_inverse_u8(const b200dct_plan *pl);
bool stream_capturing(cudaStream_t s);
bool pdl_enabled(bool capturing); // programmatic dependent launch for a launch (never on a capturing stream)
}
