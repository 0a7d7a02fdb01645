// host_pipeline.cu -- host-buffer round trips: what the reference's main() does around its two
// calls (cudaMalloc, H2D, dct, idct, D2H: main_newAppr.cu:88-124) as a chunked, overlapped
// pipeline on top of the device entry point b200dct_roundtrip.
//
// An image is cut into block-row chunks (every chunk is itself a valid image: blocks are
// independent); chunk c goes to slot c % NSLOT, and every slot owns a stream and an input and an
// output device buffer: H2D -> fused kernel -> D2H are stream-ordered inside a slot and overlap
// across slots (both copy engines and the SMs busy at once).  The slot ring simply carries on
// from one image to the next, so consecutive submissions overlap as well: image i+1 is uploading
// while image i is still on its way back -- no fill/drain bubble per image.
#include <cuda_runtime.h>
#include <stdlib.h>

#include <new>

#include "plan_internal.h"

namespace {
constexpr int MAX_SLOTS = 8;
constexpr int IMAGE_RING = 256; // completion events of the most recent submissions
}

struct b200dct_host_pipeline {
    int dev = -1;
    int nslot = 0;
    size_t chunk_bytes = 0;
    cudaStream_t st[MAX_SLOTS] = {};
    cudaEvent_t slot_done[MAX_SLOTS] = {};
    void *din[MAX_SLOTS] = {};
    void *dout[MAX_SLOTS] = {};
    cudaStream_t join = nullptr;          // orders the per-image completion events
    cudaEvent_t image_done[IMAGE_RING] = {};
    unsigned long long submitted = 0;     // images submitted so far (ticket of the next one)
    int next_slot = 0;
    int launches = 0;                     // kernels launched by the last submit
};

static void pipeline_free(b200dct_host_pipeline *p)
{
    // errors are ignored on purpose: at process exit the context may already be gone
    for (int i = 0; i < MAX_SLOTS; i++) {
        if (p->din[i]) cudaFree(p->din[i]);
        if (p->dout[i]) cudaFree(p->dout[i]);
        if (p->slot_done[i]) cudaEventDestroy(p->slot_done[i]);
        if (p->st[i]) cudaStreamDestroy(p->st[i]);
    }
    for (int i = 0; i < IMAGE_RING; i++)
        if (p->image_done[i]) cudaEventDestroy(p->image_done[i]);
    if (p->join) cudaStreamDestroy(p->join);
    (void)cudaGetLastError();
}

// Chunk sizes, measured on B200 / PCIe Gen5 (H2D alone 55.5 GB/s, D2H alone 56.3, both at once
// 48.7 each way; profiles/r02_e2e_pipeline.txt, 8192^2 f32 = 256 MiB each way per image):
//  * one image per call (synchronous form): every call pays one chunk of fill and one of drain, so
//    chunks must be small -- 16 MiB x 4 slots: 6.16 ms (2..32 MiB tried in round 1);
//  * a sequence of images through a pipeline object: no per-image bubble, so large chunks win --
//    4 MiB 7.2 ms, 8: 6.4, 16: 5.89, 32: 5.65, 64 MiB x 3 slots: 5.55 ms = 48.4 GB/s each way =
//    0.99 of the duplex ceiling (u8 images: 1.44 ms).
static size_t env_mb(const char *name, int dflt)
{
    const char *e = getenv(name);
    const int mb = (e && atoi(e) >= 1 && atoi(e) <= 1024) ? atoi(e) : dflt;
    return (size_t)mb << 20;
}
static size_t default_chunk_bytes() { return env_mb("B200DCT_HOST_CHUNK_MB", 16); }      // synchronous call
static size_t default_pipeline_chunk_bytes() { return env_mb("B200DCT_PIPE_CHUNK_MB", 64); } // pipeline objects

extern "C" int b200dct_host_pipeline_create(b200dct_host_pipeline **out, size_t chunk_bytes, int slots)
{
    if (!out) return B200DCT_ERR_ARG;
    *out = nullptr;
    if (slots == 0) slots = 3;
    if (slots < 2 || slots > MAX_SLOTS) return B200DCT_ERR_ARG;
    if (chunk_bytes == 0) chunk_bytes = default_pipeline_chunk_bytes();
    chunk_bytes = (chunk_bytes + 255) & ~(size_t)255;
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess) return B200DCT_ERR_NODEVICE;
    b200dct_host_pipeline *p = new (std::nothrow) b200dct_host_pipeline;
    if (!p) return B200DCT_ERR_NOMEM;
    p->dev = dev;
    p->nslot = slots;
    p->chunk_bytes = chunk_bytes;
    bool ok = cudaStreamCreateWithFlags(&p->join, cudaStreamNonBlocking) == cudaSuccess;
    for (int i = 0; ok && i < slots; i++)
        ok = cudaStreamCreateWithFlags(&p->st[i], cudaStreamNonBlocking) == cudaSuccess &&
             cudaEventCreateWithFlags(&p->slot_done[i], cudaEventDisableTiming) == cudaSuccess &&
             cudaMalloc(&p->din[i], chunk_bytes) == cudaSuccess && cudaMalloc(&p->dout[i], chunk_bytes) == cudaSuccess;
    for (int i = 0; ok && i < IMAGE_RING; i++) ok = cudaEventCreateWithFlags(&p->image_done[i], cudaEventDisableTiming) == cudaSuccess;
    if (!ok) {
        pipeline_free(p);
        delete p;
        return cudaGetDeviceCount(&dev) == cudaSuccess ? B200DCT_ERR_NOMEM : B200DCT_ERR_NODEVICE;
    }
    *out = p;
    return B200DCT_OK;
}

extern "C" void b200dct_host_pipeline_destroy(b200dct_host_pipeline *p)
{
    if (!p) return;
    int cur = -1;
    const bool sw = cudaGetDevice(&cur) == cudaSuccess && cur != p->dev && cudaSetDevice(p->dev) == cudaSuccess;
    for (int i = 0; i < p->nslot; i++)
        if (p->st[i]) cudaStreamSynchronize(p->st[i]);
    pipeline_free(p);
    if (sw) cudaSetDevice(cur);
    delete p;
}

extern "C" size_t b200dct_host_pipeline_chunk_bytes(const b200dct_host_pipeline *p) { return p ? p->chunk_bytes : 0; }

extern "C" int b200dct_host_pipeline_submit(b200dct_host_pipeline *p, const b200dct_plan *plan, const void *h_in,
                                            b200dct_dtype in_dt, void *h_out, b200dct_dtype out_dt, int H, int W,
                                            unsigned long long *ticket_or_null)
{
    if (!p || !plan || !h_in || !h_out) return B200DCT_ERR_ARG;
    if (!b200dct::whole_blocks(H, W)) return B200DCT_ERR_SHAPE;
    if (in_dt != out_dt || (in_dt != B200DCT_F32 && in_dt != B200DCT_U8)) return B200DCT_ERR_ARG;
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess) return B200DCT_ERR_NODEVICE;
    if (dev != p->dev) return B200DCT_ERR_ARG; // a pipeline belongs to the device it was created on
    const size_t es = in_dt == B200DCT_F32 ? 4 : 1;
    const size_t row = (size_t)W * es;
    long long rows = (long long)(p->chunk_bytes / row) & ~7ll;
    if (rows < 8) return B200DCT_ERR_SHAPE; // one block-row does not fit a chunk: create the pipeline with larger chunks
    if (rows > H) rows = H;

    int launches = 0, rc = B200DCT_OK;
    unsigned used = 0;
    for (long long r0 = 0; r0 < H; r0 += rows) {
        const int slot = p->next_slot;
        p->next_slot = (p->next_slot + 1) % p->nslot;
        const int h = (int)((H - r0) < rows ? (H - r0) : rows);
        const size_t bytes = (size_t)h * row;
        cudaStream_t s = p->st[slot];
        cudaError_t e = cudaMemcpyAsync(p->din[slot], (const char *)h_in + (size_t)r0 * row, bytes, cudaMemcpyHostToDevice, s);
        if (e != cudaSuccess) { rc = (int)e; break; }
        rc = b200dct_roundtrip(plan, p->din[slot], in_dt, row, p->dout[slot], out_dt, row, nullptr, B200DCT_F32, 0, h, W, s);
        if (rc != B200DCT_OK) break;
        launches += b200dct_last_launch_count();
        e = cudaMemcpyAsync((char *)h_out + (size_t)r0 * row, p->dout[slot], bytes, cudaMemcpyDeviceToHost, s);
        if (e != cudaSuccess) { rc = (int)e; break; }
        used |= 1u << slot;
    }
    // completion of this image = the last chunk of every slot it used; funnel them into one event
    for (int i = 0; i < p->nslot; i++) {
        if (!(used & (1u << i))) continue;
        cudaError_t e = cudaEventRecord(p->slot_done[i], p->st[i]);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(p->join, p->slot_done[i], 0);
        if (e != cudaSuccess && rc == B200DCT_OK) rc = (int)e;
    }
    const unsigned long long ticket = p->submitted++;
    cudaError_t e = cudaEventRecord(p->image_done[ticket % IMAGE_RING], p->join);
    if (e != cudaSuccess && rc == B200DCT_OK) rc = (int)e;
    if (ticket_or_null) *ticket_or_null = ticket;
    p->launches = launches;
    return rc;
}

extern "C" int b200dct_host_pipeline_wait(b200dct_host_pipeline *p, unsigned long long ticket)
{
    if (!p || ticket >= p->submitted) return B200DCT_ERR_ARG;
    // events complete in submission order (they are recorded on one stream), so for a ticket that has
    // left the ring the oldest event still in the ring is a later one: waiting for it is sufficient
    unsigned long long t = ticket;
    if (p->submitted - t > IMAGE_RING) t = p->submitted - IMAGE_RING;
    const cudaError_t e = cudaEventSynchronize(p->image_done[t % IMAGE_RING]);
    return e == cudaSuccess ? B200DCT_OK : (int)e;
}

extern "C" int b200dct_host_pipeline_drain(b200dct_host_pipeline *p)
{
    if (!p) return B200DCT_ERR_ARG;
    int rc = B200DCT_OK;
    for (int i = 0; i < p->nslot; i++) {
        const cudaError_t e = cudaStreamSynchronize(p->st[i]);
        if (e != cudaSuccess && rc == B200DCT_OK) rc = (int)e;
    }
    const cudaError_t e = cudaStreamSynchronize(p->join);
    if (e != cudaSuccess && rc == B200DCT_OK) rc = (int)e;
    return rc;
}

extern "C" int b200dct_host_pipeline_last_launch_count(const b200dct_host_pipeline *p) { return p ? p->launches : 0; }

// ------------------------------------------------------------------ the synchronous one-call form
// One pipeline per calling thread and device, created on first use and destroyed with the thread
// (or by b200dct_host_release()): short-lived worker threads do not accumulate streams and device
// buffers (round 1 leaked them until the context died).
namespace {
struct ThreadPipe {
    b200dct_host_pipeline *p = nullptr;
    ~ThreadPipe() { b200dct_host_pipeline_destroy(p); }
};
thread_local ThreadPipe tl_pipe;
thread_local int tl_host_launches = 0;
}

extern "C" int b200dct_host_release(void)
{
    b200dct_host_pipeline_destroy(tl_pipe.p);
    tl_pipe.p = nullptr;
    return B200DCT_OK;
}

extern "C" int b200dct_roundtrip_host(const b200dct_plan *plan, const void *h_in, b200dct_dtype in_dt, void *h_out,
                                      b200dct_dtype out_dt, int H, int W)
{
    tl_host_launches = 0;
    if (!plan || !h_in || !h_out) return B200DCT_ERR_ARG;
    if (!b200dct::whole_blocks(H, W)) return B200DCT_ERR_SHAPE;
    if (in_dt != out_dt || (in_dt != B200DCT_F32 && in_dt != B200DCT_U8)) return B200DCT_ERR_ARG;
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess) return B200DCT_ERR_NODEVICE;
    const size_t row8 = (size_t)W * (in_dt == B200DCT_F32 ? 4 : 1) * 8; // one block-row must fit a chunk
    size_t want = default_chunk_bytes();
    if (want < row8) want = row8;
    if (tl_pipe.p && (tl_pipe.p->dev != dev || tl_pipe.p->chunk_bytes < row8)) b200dct_host_release();
    if (!tl_pipe.p) {
        const int rc = b200dct_host_pipeline_create(&tl_pipe.p, want, 4);
        if (rc != B200DCT_OK) return rc;
    }
    int rc = b200dct_host_pipeline_submit(tl_pipe.p, plan, h_in, in_dt, h_out, out_dt, H, W, nullptr);
    const int rc2 = b200dct_host_pipeline_drain(tl_pipe.p);
    tl_host_launches = tl_pipe.p->launches;
    return rc != B200DCT_OK ? rc : rc2;
}

extern "C" int b200dct_host_last_launch_count(void) { return tl_host_launches; }
