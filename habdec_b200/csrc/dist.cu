// NCCL transport of the result gather (SURVEY.md 8e): every rank packs one hbd_result_record per local channel
// (hbd_pack_results), ranks > 0 ncclSend them to rank 0, rank 0 ncclRecv's them straight into one device buffer, copies
// it to pinned host memory and feeds its hbd_result_sink.  No collective touches the signal path.
//
// NCCL is bound at run time (dlopen "libnccl.so.2"): the library has no link-time dependency on it, stays loadable on a
// single-GPU box without NCCL, and inside a process that already carries an NCCL (torch's bundled one) the same copy is
// used.  Only the long-stable part of the NCCL API is touched.
#include "../../include/habdec_b200.h"
#include "api_internal.h"
#include "cuda_res.h"

#include <cuda_runtime.h>
#include <dlfcn.h>

#include <cstring>
#include <mutex>
#include <string>
#include <vector>

namespace {

struct NcclUid { char internal[128]; };            // ncclUniqueId (NCCL_UNIQUE_ID_BYTES = 128), passed by value
typedef int ncclResult;                            // ncclSuccess == 0
typedef void* ncclComm;
enum { kNcclInt8 = 0, kNcclInt32 = 2 };            // ncclInt8 / ncclChar = 0, ncclInt32 / ncclInt = 2

struct NcclApi {
    void* lib = nullptr;
    ncclResult (*GetUniqueId)(NcclUid*) = nullptr;
    ncclResult (*CommInitRank)(ncclComm*, int, NcclUid, int) = nullptr;
    ncclResult (*CommDestroy)(ncclComm) = nullptr;
    ncclResult (*Send)(const void*, size_t, int, int, ncclComm, cudaStream_t) = nullptr;
    ncclResult (*Recv)(void*, size_t, int, int, ncclComm, cudaStream_t) = nullptr;
    ncclResult (*AllGather)(const void*, void*, size_t, int, ncclComm, cudaStream_t) = nullptr;
    ncclResult (*GroupStart)() = nullptr;
    ncclResult (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult) = nullptr;
    std::string err;
};

NcclApi* nccl_api()
{
    static NcclApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        for (const char* name : {"libnccl.so.2", "libnccl.so"}) {
            api.lib = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
            if (api.lib) break;
        }
        if (!api.lib) { api.err = std::string("NCCL not found: ") + (dlerror() ? dlerror() : "dlopen failed"); return; }
        auto sym = [&](const char* n) { void* p = dlsym(api.lib, n); if (!p && api.err.empty()) api.err = std::string("NCCL symbol missing: ") + n; return p; };
        api.GetUniqueId = reinterpret_cast<decltype(api.GetUniqueId)>(sym("ncclGetUniqueId"));
        api.CommInitRank = reinterpret_cast<decltype(api.CommInitRank)>(sym("ncclCommInitRank"));
        api.CommDestroy = reinterpret_cast<decltype(api.CommDestroy)>(sym("ncclCommDestroy"));
        api.Send = reinterpret_cast<decltype(api.Send)>(sym("ncclSend"));
        api.Recv = reinterpret_cast<decltype(api.Recv)>(sym("ncclRecv"));
        api.AllGather = reinterpret_cast<decltype(api.AllGather)>(sym("ncclAllGather"));
        api.GroupStart = reinterpret_cast<decltype(api.GroupStart)>(sym("ncclGroupStart"));
        api.GroupEnd = reinterpret_cast<decltype(api.GroupEnd)>(sym("ncclGroupEnd"));
        api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(sym("ncclGetErrorString"));
    });
    return &api;
}

struct DistCtx {
    int rank = 0, world = 1;
    ncclComm comm = nullptr;
    bool own_comm = false;
    hbd::Stream stream;                        // declared before the buffers and events, so it is destroyed after them
    std::vector<int> counts, offsets;          // channels per rank, first record of every rank in the gathered buffer
    int total = 0;
    // A gather must not stall the thread that also feeds the GPU: senders enqueue and return (their buffers rotate through
    // a pool of kPool slots, a slot is reused once its send has completed), and rank 0 hands its pinned receive buffer to
    // the sink WITHOUT copying (hbd::sink_feed_borrowed); the sink is flushed before that slot comes round again.
    static constexpr int kPool = 4;
    hbd::HostPtr<hbd_result_record> h_send[kPool];   // pinned, counts[rank] records each
    hbd::DevPtr<hbd_result_record> d_send[kPool];
    hbd::Event ev_sent[kPool];
    hbd::DevPtr<hbd_result_record> d_recv;     // rank 0: total records
    hbd::HostPtr<hbd_result_record> h_recv[kPool];   // rank 0: pinned, total records each
    hbd_result_sink* fed[kPool] = {};          // the sink that borrowed slot k
    hbd::DevPtr<int> d_cnt;
    unsigned long long gathers = 0;
    // the steps that must come before the members release themselves: nothing in flight on the stream, the owned
    // communicator destroyed, every sink that borrows a pinned receive buffer flushed
    ~DistCtx()
    {
        if (stream) cudaStreamSynchronize(stream.get());
        if (own_comm && comm && nccl_api()->CommDestroy) nccl_api()->CommDestroy(comm);
        for (hbd_result_sink* f : fed) if (f) hbd::sink_flush(f);
    }
};

int fail(hbd_decoder* h, const std::string& what)
{
    hbd::internal_set_error(h, what);
    return HBD_ERR_CUDA;
}

int setup(hbd_decoder* h, DistCtx* c)
{
    NcclApi* n = nccl_api();
    const int n_ch = hbd_n_channels(h);
    if (hbd::stream_create(c->stream) != cudaSuccess) return fail(h, "dist: stream");
    // every rank learns how many channels the others own (one tiny all-gather at start-up)
    if (hbd::dev_alloc(c->d_cnt, size_t(c->world + 1)) != cudaSuccess) return fail(h, "dist: cudaMalloc");
    if (cudaMemcpyAsync(c->d_cnt.get() + c->world, &n_ch, sizeof(int), cudaMemcpyHostToDevice, c->stream.get()) != cudaSuccess) return fail(h, "dist: memcpy");
    c->counts.assign(size_t(c->world), n_ch);
    if (c->world > 1) {
        const ncclResult r = n->AllGather(c->d_cnt.get() + c->world, c->d_cnt.get(), 1, kNcclInt32, c->comm, c->stream.get());
        if (r) return fail(h, std::string("ncclAllGather: ") + n->GetErrorString(r));
        if (cudaMemcpyAsync(c->counts.data(), c->d_cnt.get(), sizeof(int) * size_t(c->world), cudaMemcpyDeviceToHost, c->stream.get()) != cudaSuccess) return fail(h, "dist: memcpy");
    }
    if (cudaStreamSynchronize(c->stream.get()) != cudaSuccess) return fail(h, "dist: all-gather of the channel counts failed");
    c->offsets.assign(size_t(c->world), 0);
    c->total = 0;
    for (int r = 0; r < c->world; ++r) { c->offsets[size_t(r)] = c->total; c->total += c->counts[size_t(r)]; }
    const size_t mine = size_t(n_ch), all = size_t(c->total);
    for (int k = 0; k < DistCtx::kPool; ++k) {
        if (hbd::host_alloc(c->h_send[k], mine) != cudaSuccess || hbd::dev_alloc(c->d_send[k], mine) != cudaSuccess ||
            hbd::event_create(c->ev_sent[k]) != cudaSuccess) return fail(h, "dist: buffers");
        if (c->rank == 0 && c->world > 1 && hbd::host_alloc(c->h_recv[k], all) != cudaSuccess) return fail(h, "dist: buffers");
    }
    if (c->rank == 0 && c->world > 1 && hbd::dev_alloc(c->d_recv, all) != cudaSuccess) return fail(h, "dist: buffers");
    return HBD_OK;
}

} // namespace

namespace hbd { void internal_free_dist(void* ctx) { delete static_cast<DistCtx*>(ctx); } }

extern "C" {

int hbd_dist_unique_id(unsigned char out[128])
{
    if (!out) return HBD_ERR_ARG;
    NcclApi* n = nccl_api();
    if (!n->err.empty() || !n->GetUniqueId) return HBD_ERR_STATE;
    NcclUid id;
    if (n->GetUniqueId(&id)) return HBD_ERR_CUDA;
    memcpy(out, id.internal, 128);
    return HBD_OK;
}

static int dist_attach(hbd_decoder* h, int rank, int world, ncclComm comm, bool own)
{
    hbd::DistSlot& slot = hbd::internal_dist_slot(h);
    slot.reset();
    std::unique_ptr<DistCtx> c(new DistCtx);
    c->rank = rank; c->world = world; c->comm = comm; c->own_comm = own;
    int rc = setup(h, c.get());
    if (!rc) rc = hbd_set_stats_snapshot(h, 1);   // a gather never waits for calls in flight
    if (rc) return rc;
    slot.reset(c.release());
    return HBD_OK;
}

int hbd_dist_init(hbd_decoder* h, int rank, int world, const unsigned char id[128])
{
    if (!h || world < 1 || rank < 0 || rank >= world || (world > 1 && !id)) return HBD_ERR_ARG;
    if (cudaSetDevice(hbd::internal_device(h)) != cudaSuccess) return HBD_ERR_CUDA;
    ncclComm comm = nullptr;
    if (world > 1) {
        NcclApi* n = nccl_api();
        if (!n->err.empty()) { hbd::internal_set_error(h, n->err); return HBD_ERR_STATE; }
        NcclUid uid; memcpy(uid.internal, id, 128);
        const ncclResult r = n->CommInitRank(&comm, world, uid, rank);
        if (r) return fail(h, std::string("ncclCommInitRank: ") + n->GetErrorString(r));
    }
    return dist_attach(h, rank, world, comm, true);
}

// adopt a communicator the application already has (ncclComm_t); it is not destroyed by the library
int hbd_dist_use_comm(hbd_decoder* h, void* nccl_comm, int rank, int world)
{
    if (!h || world < 1 || rank < 0 || rank >= world || (world > 1 && !nccl_comm)) return HBD_ERR_ARG;
    if (cudaSetDevice(hbd::internal_device(h)) != cudaSuccess) return HBD_ERR_CUDA;
    if (world > 1 && !nccl_api()->err.empty()) { hbd::internal_set_error(h, nccl_api()->err); return HBD_ERR_STATE; }
    return dist_attach(h, rank, world, nccl_comm, false);
}

int hbd_dist_finalize(hbd_decoder* h)
{
    if (!h) return HBD_ERR_ARG;
    hbd::DistSlot& slot = hbd::internal_dist_slot(h);
    if (slot) { cudaSetDevice(hbd::internal_device(h)); slot.reset(); }   // flushes the sinks it fed
    return HBD_OK;
}

int hbd_dist_total_channels(hbd_decoder* h)
{
    if (!h) return 0;
    DistCtx* c = static_cast<DistCtx*>(hbd::internal_dist_slot(h).get());
    return c ? c->total : hbd_n_channels(h);
}

// Every rank calls this at the same points of its call sequence.  Packs what the local channels decoded since the previous
// gather (what hbd_collect* has been through), moves the records to rank 0 and feeds `sink` there (ignored elsewhere).
// Global channel number = first channel of the rank (ranks in order) + local index.  Returns records moved or < 0.
int hbd_gather_results(hbd_decoder* h, hbd_result_sink* sink)
{
    if (!h) return HBD_ERR_ARG;
    DistCtx* c = static_cast<DistCtx*>(hbd::internal_dist_slot(h).get());
    if (!c) { hbd::internal_set_error(h, "hbd_gather_results: call hbd_dist_init first"); return HBD_ERR_STATE; }
    if (c->rank == 0 && !sink) return HBD_ERR_ARG;
    if (cudaSetDevice(hbd::internal_device(h)) != cudaSuccess) return HBD_ERR_CUDA;
    NcclApi* n = nccl_api();
    const int mine = c->counts[size_t(c->rank)];
    const int k = int(c->gathers % DistCtx::kPool);
    // slot k comes round again: its send has long completed; a sink that still borrows it takes its records in now
    if (c->gathers >= DistCtx::kPool && cudaEventSynchronize(c->ev_sent[k].get()) != cudaSuccess) return fail(h, "gather: earlier send failed");
    if (c->fed[k]) { hbd::sink_flush(c->fed[k]); c->fed[k] = nullptr; }
    const size_t got = hbd_pack_results(h, c->offsets[size_t(c->rank)], c->h_send[k].get(), size_t(mine));
    if (got != size_t(mine)) return HBD_ERR_STATE;
    const size_t rec = sizeof(hbd_result_record);
    if (c->world > 1) {
        if (c->rank != 0) {
            // enqueue and return: nothing here waits for rank 0 (which may be busy draining its own channels)
            if (cudaMemcpyAsync(c->d_send[k].get(), c->h_send[k].get(), rec * size_t(mine), cudaMemcpyHostToDevice, c->stream.get()) != cudaSuccess) return fail(h, "gather: H2D");
            const ncclResult r = n->Send(c->d_send[k].get(), rec * size_t(mine), kNcclInt8, 0, c->comm, c->stream.get());
            if (r) return fail(h, std::string("ncclSend: ") + n->GetErrorString(r));
            if (cudaEventRecord(c->ev_sent[k].get(), c->stream.get()) != cudaSuccess) return fail(h, "gather: event");
        } else {
            ncclResult r = n->GroupStart();
            for (int p = 1; p < c->world && !r; ++p)
                r = n->Recv(c->d_recv.get() + c->offsets[size_t(p)], rec * size_t(c->counts[size_t(p)]), kNcclInt8, p, c->comm, c->stream.get());
            if (!r) r = n->GroupEnd();
            if (r) return fail(h, std::string("ncclRecv: ") + n->GetErrorString(r));
            if (cudaMemcpyAsync(c->h_recv[k].get() + mine, c->d_recv.get() + mine, rec * size_t(c->total - mine), cudaMemcpyDeviceToHost, c->stream.get()) != cudaSuccess)
                return fail(h, "gather: D2H");
            if (cudaEventRecord(c->ev_sent[k].get(), c->stream.get()) != cudaSuccess) return fail(h, "gather: event");
            if (cudaStreamSynchronize(c->stream.get()) != cudaSuccess) return fail(h, "gather: transfer failed");
        }
    }
    ++c->gathers;
    if (c->rank != 0) {   // a sink on another rank mirrors that rank's own channels (same global numbering)
        if (sink) { const int rc = hbd::sink_feed_borrowed(sink, c->h_send[k].get(), size_t(mine)); if (rc) return rc; c->fed[k] = sink; }
        return mine;
    }
    int rc = hbd::sink_feed_borrowed(sink, c->h_send[k].get(), size_t(mine));
    if (c->world > 1 && !rc) rc = hbd::sink_feed_borrowed(sink, c->h_recv[k].get() + mine, size_t(c->total - mine));
    c->fed[k] = sink;
    return rc ? rc : c->total;
}

} // extern "C"
