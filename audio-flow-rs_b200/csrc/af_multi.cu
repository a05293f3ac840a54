// af_multi.cu -- multi-GPU behind the C ABI (SURVEY 8(e)): stream sharding over the GPUs of one box and the gather
// of per-stream VAD results with NCCL over NVLink.  Streams are independent (no cross-stream state anywhere in
// resampler.rs / vad.rs), so the data path has no collective.  The gather is off the critical path: the VAD scan of a
// shard writes its states straight into the rank's slot of a double-buffered gather buffer, an event hands the buffer
// to the side stream, ONE in-place ncclAllGather runs there, and the next batch on the compute stream never waits for it.
//
// NCCL is bound at run time (dlopen "libnccl.so.2"): a process that already carries one (PyTorch bundles its own) shares
// it, a plain C / Rust host gets the system library, and single-GPU use never loads it.
#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <thread>

#include "af_internal.h"

using namespace af;
using namespace afrt;

namespace {

struct NcclApi {
    void *handle = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommInitAll)(ncclComm_t *, int, const int *) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
    ncclResult_t (*GetVersion)(int *) = nullptr;
};
NcclApi g_nccl;
std::mutex g_comm_mu;

int load_nccl()
{
    if (g_nccl.handle) return AF_OK;
    // A copy the process already carries wins (PyTorch bundles its own libnccl.so.2: a process that uses both must
    // import torch BEFORE the first multi-GPU call, or torch would be handed the system library instead of its own).
    const char *names[] = {"libnccl.so.2", "libnccl.so"};
    void *h = nullptr;
    for (const char *n : names) {
        h = dlopen(n, RTLD_NOW | RTLD_NOLOAD);
        if (!h) h = dlopen(n, RTLD_NOW | RTLD_LOCAL);
        if (h) break;
    }
    if (!h) return fail(AF_ERR_NO_DEVICE, "NCCL is not available (%s): the multi-GPU entry points need libnccl.so.2", dlerror());
#define AF_SYM(field, name)                                                                   \
    g_nccl.field = reinterpret_cast<decltype(g_nccl.field)>(dlsym(h, name));                  \
    if (!g_nccl.field) { dlclose(h); return fail(AF_ERR_NO_DEVICE, "libnccl has no symbol %s", name); }
    AF_SYM(GetUniqueId, "ncclGetUniqueId")
    AF_SYM(CommInitRank, "ncclCommInitRank")
    AF_SYM(CommInitAll, "ncclCommInitAll")
    AF_SYM(CommDestroy, "ncclCommDestroy")
    AF_SYM(AllGather, "ncclAllGather")
    AF_SYM(GroupStart, "ncclGroupStart")
    AF_SYM(GroupEnd, "ncclGroupEnd")
    AF_SYM(GetErrorString, "ncclGetErrorString")
    AF_SYM(GetVersion, "ncclGetVersion")
#undef AF_SYM
    g_nccl.handle = h;
    return AF_OK;
}

#define AF_NCCL(expr)                                                                                  \
    do {                                                                                               \
        ncclResult_t _r = (expr);                                                                      \
        if (_r != ncclSuccess) return fail(AF_ERR_CUDA, "NCCL error %s at %s:%d: %s", #expr, __FILE__, __LINE__, \
                                           g_nccl.GetErrorString(_r));                                 \
    } while (0)

// the communicator of the process: every rank it owns, with the GPU and the NCCL handle of each
struct Comm {
    bool ready = false;
    int n_ranks = 0;
    std::vector<int> ranks;          // global ranks owned by this process
    std::vector<int> devices;        // their GPUs
    std::vector<ncclComm_t> comms;
    int local_index(int rank) const
    {
        for (size_t i = 0; i < ranks.size(); ++i)
            if (ranks[i] == rank) return (int)i;
        return -1;
    }
};
Comm g_comm;

uint64_t round_up64(uint64_t v, uint64_t m) { return (v + m - 1) / m * m; }

}  // namespace

namespace afrt {
void comm_shutdown_all() { (void)af_comm_shutdown(); }
}  // namespace afrt

struct af_sharded_batch {
    af_pipeline *pipe = nullptr;
    int mem = AF_MEM_DEVICE;
    size_t n_streams = 0;
    int n_ranks = 1;
    std::vector<size_t> first;                 // n_ranks + 1
    std::vector<uint32_t> n_vad;               // per global stream
    std::vector<af_batch *> local;             // per local rank (index into g_comm.ranks)
    std::vector<int> ranks, devices;           // copies of the communicator's at creation
    uint64_t rows_max = 0, row_stride = 0;     // gather geometry: [n_ranks][rows_max][row_stride] bytes
    std::vector<DevBuf<uint8_t>> gbuf[2];      // per local rank, double buffered
    std::vector<cudaEvent_t> ev_compute[2], ev_gather_begin[2], ev_gather_end[2];
    std::vector<bool> gathered_once[2];
    uint64_t steps = 0;
    int last_parity = -1;                      // buffer of the last run with a gather
};

extern "C" {

AF_API int af_comm_size(void) { return g_comm.ready ? g_comm.n_ranks : 0; }

AF_API int af_comm_shutdown(void)
{
    std::lock_guard<std::mutex> lk(g_comm_mu);
    if (!g_comm.ready) return AF_OK;
    for (size_t i = 0; i < g_comm.comms.size(); ++i) {
        if (!g_comm.comms[i]) continue;
        DevScope scope_(g_comm.devices[i]);
        cudaDeviceSynchronize();
        g_nccl.CommDestroy(g_comm.comms[i]);
    }
    g_comm = Comm{};
    return AF_OK;
}

AF_API int af_init_multi(int n_gpus)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        (void)cudaGetLastError();
        return fail(AF_ERR_NO_DEVICE, "no CUDA device available; libaudioflow_gpu has no CPU fallback");
    }
    if (n_gpus <= 0) n_gpus = n;
    if (n_gpus > n || n_gpus > AF_MAX_GPUS) return fail(AF_ERR_INVALID, "%d GPUs requested, %d present (max %d)", n_gpus, n, AF_MAX_GPUS);
    for (int d = 0; d < n_gpus; ++d) {
        int rc = init_device(d);
        if (rc) return rc;
    }
    int rc = af_init(0);
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(g_comm_mu);
    if (g_comm.ready) {
        if (g_comm.n_ranks == n_gpus && (int)g_comm.ranks.size() == n_gpus) return AF_OK;
        return fail(AF_ERR_INVALID, "a communicator of %d ranks already exists (af_comm_shutdown first)", g_comm.n_ranks);
    }
    Comm c;
    c.n_ranks = n_gpus;
    for (int d = 0; d < n_gpus; ++d) { c.ranks.push_back(d); c.devices.push_back(d); }
    c.comms.assign(n_gpus, nullptr);
    if (n_gpus > 1) {
        rc = load_nccl();
        if (rc) return rc;
        // peer access for direct loads / stores between the GPUs of the process (NCCL sets up its own paths)
        for (int a = 0; a < n_gpus; ++a) {
            DevScope scope_(a);
            for (int b = 0; b < n_gpus; ++b) {
                if (a == b) continue;
                int can = 0;
                if (cudaDeviceCanAccessPeer(&can, a, b) == cudaSuccess && can) {
                    cudaError_t pe = cudaDeviceEnablePeerAccess(b, 0);
                    if (pe != cudaSuccess) (void)cudaGetLastError();          // already enabled is fine
                }
            }
        }
        AF_NCCL(g_nccl.CommInitAll(c.comms.data(), n_gpus, c.devices.data()));
    }
    c.ready = true;
    g_comm = c;
    return AF_OK;
}

AF_API int af_comm_unique_id(uint8_t id[128])
{
    if (!id) return fail(AF_ERR_INVALID, "null id");
    int rc = load_nccl();
    if (rc) return rc;
    static_assert(NCCL_UNIQUE_ID_BYTES == 128, "the C ABI carries the NCCL unique id as 128 bytes");
    ncclUniqueId u;
    AF_NCCL(g_nccl.GetUniqueId(&u));
    memcpy(id, u.internal, 128);
    return AF_OK;
}

AF_API int af_comm_init_rank(int n_ranks, int rank, const uint8_t id[128])
{
    if (n_ranks <= 0 || n_ranks > AF_MAX_GPUS || rank < 0 || rank >= n_ranks) return fail(AF_ERR_INVALID, "bad rank %d of %d", rank, n_ranks);
    int rc = require_ctx();
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(g_comm_mu);
    if (g_comm.ready) return fail(AF_ERR_INVALID, "a communicator of %d ranks already exists (af_comm_shutdown first)", g_comm.n_ranks);
    Comm c;
    c.n_ranks = n_ranks;
    c.ranks.push_back(rank); c.devices.push_back(cur_device());
    c.comms.assign(1, nullptr);
    if (n_ranks > 1) {
        if (!id) return fail(AF_ERR_INVALID, "null id");
        rc = load_nccl();
        if (rc) return rc;
        ncclUniqueId u;
        memcpy(u.internal, id, 128);
        AF_NCCL(g_nccl.CommInitRank(&c.comms[0], n_ranks, u, rank));
    }
    c.ready = true;
    g_comm = c;
    return AF_OK;
}

AF_API int af_shard_partition(const af_stream_desc *streams, size_t n_streams, int n_shards, size_t *first)
{
    if ((!streams && n_streams) || !first || n_shards <= 0) return fail(AF_ERR_INVALID, "bad argument");
    // prefix costs in bytes of input; boundary r is where the prefix comes closest to r / n_shards of the total
    std::vector<double> cum(n_streams + 1, 0.0);
    for (size_t i = 0; i < n_streams; ++i)
        cum[i + 1] = cum[i] + (double)streams[i].n_samples * (streams[i].format == AF_FMT_I16 ? 2.0 : 4.0);
    const double total = cum[n_streams];
    first[0] = 0;
    for (int r = 1; r < n_shards; ++r) {
        const double target = total * (double)r / (double)n_shards;
        size_t i = (size_t)(std::lower_bound(cum.begin(), cum.end(), target) - cum.begin());
        if (i > n_streams) i = n_streams;
        if (i > 0 && std::fabs(cum[i - 1] - target) <= std::fabs(cum[i] - target)) --i;
        first[r] = std::min(std::max(i, first[r - 1]), n_streams);
    }
    first[n_shards] = n_streams;
    return AF_OK;
}

AF_API void af_sharded_batch_destroy(af_sharded_batch *b)
{
    if (!b) return;
    for (size_t li = 0; li < b->local.size(); ++li) {
        DevScope scope_(b->devices[li]);
        cudaDeviceSynchronize();
        for (int p = 0; p < 2; ++p) {
            if (li < b->gbuf[p].size()) b->gbuf[p][li].reset();
            if (li < b->ev_compute[p].size() && b->ev_compute[p][li]) cudaEventDestroy(b->ev_compute[p][li]);
            if (li < b->ev_gather_begin[p].size() && b->ev_gather_begin[p][li]) cudaEventDestroy(b->ev_gather_begin[p][li]);
            if (li < b->ev_gather_end[p].size() && b->ev_gather_end[p][li]) cudaEventDestroy(b->ev_gather_end[p][li]);
        }
        if (b->local[li]) af_batch_destroy(b->local[li]);
    }
    delete b;
}

AF_API int af_sharded_batch_create(af_pipeline *p, const af_stream_desc *streams, size_t n_streams, int mem,
                                   af_sharded_batch **out)
{
    if (!p || !out || (!streams && n_streams)) return fail(AF_ERR_INVALID, "null argument");
    if (mem != AF_MEM_DEVICE && mem != AF_MEM_HOST) return fail(AF_ERR_INVALID, "bad memory kind %d", mem);
    if (!g_comm.ready) {                                   // no communicator: a single rank on the thread's GPU
        int rc = af_comm_init_rank(1, 0, nullptr);
        if (rc) return rc;
    }
    std::unique_ptr<af_sharded_batch, void (*)(af_sharded_batch *)> b(new af_sharded_batch, af_sharded_batch_destroy);
    b->pipe = p; b->mem = mem; b->n_streams = n_streams; b->n_ranks = g_comm.n_ranks;
    b->ranks = g_comm.ranks; b->devices = g_comm.devices;
    b->first.assign(b->n_ranks + 1, 0);
    int rc = af_shard_partition(streams, n_streams, b->n_ranks, b->first.data());
    if (rc) return rc;
    // every rank plans every stream's frame count: the rows of the gathered result need no exchange of sizes
    const af_pipeline_config &cfg = pipeline_cfg(p);
    b->n_vad.assign(n_streams, 0);
    uint64_t max_vad = 0;
    for (size_t i = 0; i < n_streams; ++i) {
        rc = plan_stream_counts(cfg, streams[i], nullptr, nullptr, &b->n_vad[i]);
        if (rc) return rc;
        max_vad = std::max<uint64_t>(max_vad, b->n_vad[i]);
    }
    for (int r = 0; r < b->n_ranks; ++r) b->rows_max = std::max<uint64_t>(b->rows_max, b->first[r + 1] - b->first[r]);
    b->row_stride = round_up64(std::max<uint64_t>(max_vad, 16), 16);
    const size_t n_local = b->ranks.size();
    b->local.assign(n_local, nullptr);
    for (int q = 0; q < 2; ++q) {
        b->gbuf[q].resize(n_local);
        b->ev_compute[q].assign(n_local, nullptr);
        b->ev_gather_begin[q].assign(n_local, nullptr);
        b->ev_gather_end[q].assign(n_local, nullptr);
        b->gathered_once[q].assign(n_local, false);
    }
    for (size_t li = 0; li < n_local; ++li) {
        const int r = b->ranks[li];
        AF_SCOPE(b->devices[li]);
        const size_t lo = b->first[r], cnt = b->first[r + 1] - lo;
        rc = af_batch_create(p, streams + lo, cnt, mem, &b->local[li]);
        if (rc) return rc;
        if (batch_device(b->local[li]) != b->devices[li])
            return fail(AF_ERR_INVALID, "the streams of rank %d live on GPU %d, the rank runs on GPU %d", r, batch_device(b->local[li]), b->devices[li]);
        if (cfg.vad_enable && mem == AF_MEM_DEVICE) {
            const size_t bytes = std::max<size_t>((size_t)b->n_ranks * b->rows_max * b->row_stride, 256);
            for (int q = 0; q < 2; ++q) {
                AF_CUDA(b->gbuf[q][li].alloc(bytes));
                AF_CUDA(cudaMemset(b->gbuf[q][li].get(), 0, bytes));
                AF_CUDA(cudaEventCreateWithFlags(&b->ev_compute[q][li], cudaEventDisableTiming));
                AF_CUDA(cudaEventCreate(&b->ev_gather_begin[q][li]));
                AF_CUDA(cudaEventCreate(&b->ev_gather_end[q][li]));
            }
        }
    }
    *out = b.release();
    return AF_OK;
}

AF_API int af_sharded_batch_shard(const af_sharded_batch *b, int rank, size_t *first, size_t *count, int *device)
{
    if (!b || rank < 0 || rank >= b->n_ranks) return fail(AF_ERR_INVALID, "bad rank");
    if (first) *first = b->first[rank];
    if (count) *count = b->first[rank + 1] - b->first[rank];
    if (device) {
        *device = -1;
        for (size_t li = 0; li < b->ranks.size(); ++li)
            if (b->ranks[li] == rank) *device = b->devices[li];
    }
    return AF_OK;
}

AF_API af_batch *af_sharded_batch_local(af_sharded_batch *b, int rank)
{
    if (!b) return nullptr;
    for (size_t li = 0; li < b->ranks.size(); ++li)
        if (b->ranks[li] == rank) return b->local[li];
    return nullptr;
}

AF_API int af_sharded_batch_wait(af_sharded_batch *b)
{
    if (!b) return fail(AF_ERR_INVALID, "null batch");
    for (size_t li = 0; li < b->local.size(); ++li) {
        AF_SCOPE(b->devices[li]);
        AF_CUDA(cudaStreamSynchronize(cur_ctx().stream));
        AF_CUDA(cudaStreamSynchronize(cur_ctx().side));
    }
    return AF_OK;
}

AF_API int af_sharded_batch_join(af_sharded_batch *b)
{
    if (!b) return fail(AF_ERR_INVALID, "null batch");
    if (b->last_parity < 0) return AF_OK;
    for (size_t li = 0; li < b->local.size(); ++li) {
        if (!b->gathered_once[b->last_parity][li]) continue;
        AF_SCOPE(b->devices[li]);
        AF_CUDA(cudaStreamWaitEvent(cur_ctx().stream, b->ev_gather_end[b->last_parity][li], 0));
    }
    return AF_OK;
}

AF_API int af_sharded_batch_run(af_sharded_batch *b, const af_sharded_outputs *out, int gather, int async)
{
    if (!b || !out) return fail(AF_ERR_INVALID, "null argument");
    if (b->mem != AF_MEM_DEVICE) return fail(AF_ERR_INVALID, "batch was planned for host buffers; use af_sharded_batch_run_host");
    const af_pipeline_config &cfg = pipeline_cfg(b->pipe);
    const bool do_gather = gather != 0 && cfg.vad_enable && b->n_streams > 0;
    const int par = (int)(b->steps & 1u);
    const size_t n_local = b->local.size();
    const size_t slot_bytes = (size_t)b->rows_max * b->row_stride;
    for (size_t li = 0; li < n_local; ++li) {
        int rc = batch_check_outputs(b->local[li], &out->shard[b->ranks[li]]);
        if (rc) return rc;
    }
    // ---- compute: every local GPU gets its kernels before anything waits ----
    for (size_t li = 0; li < n_local; ++li) {
        const int r = b->ranks[li];
        AF_SCOPE(b->devices[li]);
        cudaStream_t st = cur_ctx().stream;
        const af_outputs *o = &out->shard[r];
        if (do_gather) {
            // the gather that used this buffer two runs ago must have drained before the scan overwrites the slot
            if (b->gathered_once[par][li]) AF_CUDA(cudaStreamWaitEvent(st, b->ev_gather_end[par][li], 0));
            int rc = batch_run_on(b->local[li], o, b->gbuf[par][li].get() + (size_t)r * slot_bytes, b->row_stride, st);
            if (rc) return rc;
            AF_CUDA(cudaEventRecord(b->ev_compute[par][li], st));
        } else {
            int rc = batch_run_on(b->local[li], o, o->vad, o->vad_stride, st);
            if (rc) return rc;
        }
    }
    // ---- gather: one in-place all-gather per GPU on its side stream ----
    if (do_gather) {
        for (size_t li = 0; li < n_local; ++li) {
            AF_SCOPE(b->devices[li]);
            AF_CUDA(cudaStreamWaitEvent(cur_ctx().side, b->ev_compute[par][li], 0));
            AF_CUDA(cudaEventRecord(b->ev_gather_begin[par][li], cur_ctx().side));
        }
        if (b->n_ranks > 1) {
            AF_NCCL(g_nccl.GroupStart());
            for (size_t li = 0; li < n_local; ++li) {
                const int r = b->ranks[li];
                DevScope scope_(b->devices[li]);
                ncclResult_t nr = g_nccl.AllGather(b->gbuf[par][li].get() + (size_t)r * slot_bytes, b->gbuf[par][li].get(), slot_bytes, ncclUint8,
                                                   g_comm.comms[li], cur_ctx().side);
                if (nr != ncclSuccess) { g_nccl.GroupEnd(); return fail(AF_ERR_CUDA, "ncclAllGather: %s", g_nccl.GetErrorString(nr)); }
            }
            AF_NCCL(g_nccl.GroupEnd());
        }
        for (size_t li = 0; li < n_local; ++li) {
            AF_SCOPE(b->devices[li]);
            AF_CUDA(cudaEventRecord(b->ev_gather_end[par][li], cur_ctx().side));
            b->gathered_once[par][li] = true;
        }
        b->last_parity = par;
        b->steps += 1;
    }
    if (!async) return af_sharded_batch_wait(b);
    return AF_OK;
}

AF_API int af_sharded_batch_gathered(af_sharded_batch *b, int rank, const uint8_t **states, uint64_t *row_stride,
                                     uint64_t *rows_per_rank, uint32_t *n_vad_frames)
{
    if (!b) return fail(AF_ERR_INVALID, "null batch");
    const int li = [&] { for (size_t i = 0; i < b->ranks.size(); ++i) if (b->ranks[i] == rank) return (int)i; return -1; }();
    if (li < 0) return fail(AF_ERR_INVALID, "rank %d is not owned by this process", rank);
    if (b->last_parity < 0) return fail(AF_ERR_INVALID, "no run with a gather yet");
    if (states) *states = b->gbuf[b->last_parity][li].get();
    if (row_stride) *row_stride = b->row_stride;
    if (rows_per_rank) *rows_per_rank = b->rows_max;
    if (n_vad_frames) memcpy(n_vad_frames, b->n_vad.data(), b->n_vad.size() * sizeof(uint32_t));
    return AF_OK;
}

AF_API int af_sharded_batch_gathered_host(af_sharded_batch *b, int rank, uint8_t *states, uint64_t stride)
{
    if (!b || !states) return fail(AF_ERR_INVALID, "null argument");
    const int li = [&] { for (size_t i = 0; i < b->ranks.size(); ++i) if (b->ranks[i] == rank) return (int)i; return -1; }();
    if (li < 0) return fail(AF_ERR_INVALID, "rank %d is not owned by this process", rank);
    if (b->last_parity < 0) return fail(AF_ERR_INVALID, "no run with a gather yet");
    uint64_t max_vad = 0;
    for (uint32_t v : b->n_vad) max_vad = std::max<uint64_t>(max_vad, v);
    if (stride < max_vad) return fail(AF_ERR_CAPACITY, "stride %llu < %llu frames", (unsigned long long)stride, (unsigned long long)max_vad);
    AF_SCOPE(b->devices[li]);
    cudaStream_t st = cur_ctx().side;                     // ordered after the gather
    const uint8_t *g = b->gbuf[b->last_parity][li].get();
    const size_t width = (size_t)std::min<uint64_t>(stride, b->row_stride);
    for (int r = 0; r < b->n_ranks; ++r) {
        const size_t lo = b->first[r], cnt = b->first[r + 1] - lo;
        if (cnt) AF_CUDA(cudaMemcpy2DAsync(states + lo * stride, stride, g + (size_t)r * b->rows_max * b->row_stride, b->row_stride, width, cnt,
                                           cudaMemcpyDeviceToHost, st));
    }
    AF_CUDA(cudaStreamSynchronize(st));
    return AF_OK;
}

AF_API int af_sharded_batch_gather_ms(af_sharded_batch *b, int rank, float *ms)
{
    if (!b || !ms) return fail(AF_ERR_INVALID, "null argument");
    const int li = [&] { for (size_t i = 0; i < b->ranks.size(); ++i) if (b->ranks[i] == rank) return (int)i; return -1; }();
    if (li < 0 || b->last_parity < 0) return fail(AF_ERR_INVALID, "no gather on rank %d yet", rank);
    AF_SCOPE(b->devices[li]);
    AF_CUDA(cudaEventSynchronize(b->ev_gather_end[b->last_parity][li]));
    AF_CUDA(cudaEventElapsedTime(ms, b->ev_gather_begin[b->last_parity][li], b->ev_gather_end[b->last_parity][li]));
    return AF_OK;
}

AF_API int af_sharded_batch_run_host(af_sharded_batch *b, const af_outputs *o)
{
    if (!b || !o) return fail(AF_ERR_INVALID, "null argument");
    if (b->mem != AF_MEM_HOST) return fail(AF_ERR_INVALID, "batch was planned for device buffers; use af_sharded_batch_run");
    const size_t n_local = b->local.size();
    std::vector<int> rcs(n_local, AF_OK);
    std::vector<std::string> errs(n_local);
    auto work = [&](size_t li) {
        const size_t lo = b->first[b->ranks[li]];
        af_outputs sub = *o;                               // this shard's rows of the global host arrays
        if (sub.pcm) sub.pcm += lo * o->pcm_stride;
        if (sub.logmel) sub.logmel += lo * o->logmel_stride;
        if (sub.vad) sub.vad += lo * o->vad_stride;
        if (sub.energy) sub.energy += lo * o->energy_stride;
        if (sub.vad_final) sub.vad_final += lo;
        rcs[li] = af_batch_run_host(b->local[li], &sub);
        if (rcs[li] != AF_OK) {
            char buf[512];
            af_last_error(buf, sizeof(buf));
            errs[li] = buf;
        }
    };
    if (n_local == 1) work(0);
    else {
        std::vector<std::thread> th;
        for (size_t li = 0; li < n_local; ++li) th.emplace_back(work, li);   // one host thread per GPU: the copies of all GPUs overlap
        for (auto &t : th) t.join();
    }
    for (size_t li = 0; li < n_local; ++li)
        if (rcs[li] != AF_OK) return fail(rcs[li], "rank %d: %s", b->ranks[li], errs[li].c_str());
    return AF_OK;
}

}  // extern "C"
