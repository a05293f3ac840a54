// af_runtime.cu -- the C ABI of libaudioflow_gpu.so (include/audioflow_gpu.h): library context,
// compat objects mirroring the reference's Rust types, and the batched pipeline host runtime.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <map>

#include "af_internal.h"

using namespace af;
using namespace afrt;

// ------------------------------------------------------------------------------------------
// contexts: one per GPU the process uses
// ------------------------------------------------------------------------------------------
namespace afrt {

namespace {
thread_local std::string g_err;
std::atomic<uint64_t> g_launches{0};
// never destroyed: at process exit the statically linked cudart may be gone before a destructor could free anything
Context *const g_ctxs = new Context[MAX_DEV];
std::mutex g_init_mu;                 // serialises device initialisation / shutdown
std::atomic<int> g_default_dev{-1};   // the first device initialised: what a thread without a selection of its own uses
thread_local int t_dev = -1;          // the device this thread works on
std::string g_variant = "auto";
}  // namespace

int fail(int code, const char *fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

Context &cur_ctx() { return g_ctxs[t_dev >= 0 ? t_dev : 0]; }
int cur_device() { return t_dev; }
Context *device_ctx(int device) { return (device >= 0 && device < MAX_DEV && g_ctxs[device].ready) ? &g_ctxs[device] : nullptr; }
void count_launch(uint64_t n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
const std::string &kernel_variant() { return g_variant; }

int init_device(int device)
{
    std::lock_guard<std::mutex> lk(g_init_mu);
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        (void)cudaGetLastError();
        return fail(AF_ERR_NO_DEVICE, "no CUDA device available (%s); libaudioflow_gpu has no CPU fallback",
                    e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    }
    if (device < 0 || device >= n || device >= MAX_DEV) return fail(AF_ERR_INVALID, "device %d out of range (%d devices)", device, n);
    Context &c = g_ctxs[device];
    if (c.ready) return AF_OK;
    int prev = 0;
    (void)cudaGetDevice(&prev);
    struct Back { int d; ~Back() { (void)cudaSetDevice(d); } } back{prev};
    AF_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    AF_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return fail(AF_ERR_NO_DEVICE, "device %d (%s, sm_%d%d) is not a Blackwell sm_100 GPU", device, prop.name,
                    prop.major, prop.minor);
    c.sm_count = prop.multiProcessorCount;
    AF_CUDA(cudaStreamCreateWithFlags(&c.own, cudaStreamNonBlocking));
    c.stream = c.own;
    // the gather stream has the lowest priority: when a collective kernel and the next batch's fused kernel become
    // runnable together, the SMs go to the fused kernel (one persistent CTA per SM) first
    int prio_lo = 0, prio_hi = 0;
    AF_CUDA(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
    AF_CUDA(cudaStreamCreateWithPriority(&c.side, cudaStreamNonBlocking, prio_lo));
    FftTables *h = new FftTables;
    build_fft_tables(h);
    cudaError_t ce = c.d_fft.alloc(1);
    if (ce == cudaSuccess) ce = cudaMemcpy(c.d_fft.get(), h, sizeof(FftTables), cudaMemcpyHostToDevice);
    delete h;
    AF_CUDA(ce);
    c.device = device;
    c.ready = true;
    int none = -1;
    g_default_dev.compare_exchange_strong(none, device);
    return AF_OK;
}

int require_ctx()
{
    int dev = t_dev >= 0 ? t_dev : g_default_dev.load();
    if (dev < 0) {                                    // nothing initialised yet: the calling thread's current CUDA device
        int cur = 0;
        if (cudaGetDevice(&cur) != cudaSuccess) { (void)cudaGetLastError(); cur = 0; }
        dev = cur;
    }
    if (!g_ctxs[dev < MAX_DEV ? dev : 0].ready) {
        int rc = init_device(dev);
        if (rc != AF_OK) return rc;
    }
    t_dev = dev;
    AF_CUDA(cudaSetDevice(dev));
    return AF_OK;
}

DevScope::DevScope(int dev_) : prev_lib(t_dev), prev_cuda(-1), dev(dev_), rc(AF_OK)
{
    if (cudaGetDevice(&prev_cuda) != cudaSuccess) { (void)cudaGetLastError(); prev_cuda = -1; }
    if (dev < 0 || dev >= MAX_DEV || !g_ctxs[dev].ready) { rc = fail(AF_ERR_INVALID, "handle belongs to device %d, which is not initialised", dev); return; }
    t_dev = dev;
    if (prev_cuda != dev && cudaSetDevice(dev) != cudaSuccess) rc = fail(AF_ERR_CUDA, "cudaSetDevice(%d) failed", dev);
}
DevScope::~DevScope()
{
    t_dev = prev_lib;
    if (prev_cuda >= 0 && prev_cuda != dev) (void)cudaSetDevice(prev_cuda);
}

int device_of_pointer(const void *p)
{
    if (!p) return -1;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { (void)cudaGetLastError(); return -1; }
    return (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged) ? a.device : -1;
}

}  // namespace afrt

namespace {

// the context's scratch buffers grow with 25 % slack: a caller whose sizes creep up rarely reallocates
cudaError_t reserve(DevBuf<uint8_t> &b, size_t bytes) { return bytes <= b.size() ? cudaSuccess : b.alloc(bytes + bytes / 4 + 256); }

// warp-to-role layout of the fused kernel (warp_role, af_common.cuh): the V warp gets a lighter scheduler when it
// has energy chains to run.  AF_LAYOUT=<n> overrides (experiments).
uint32_t fused_layout(bool energies)
{
    static const int forced = [] { const char *e = getenv("AF_LAYOUT"); return e ? atoi(e) : -1; }();
    if (forced >= 0 && forced < N_LAYOUTS) return (uint32_t)forced;
    return energies ? 2u : 0u;
}

// exact output length of BatchResampler::process(all) + flush() and (optionally) the frac table
int plan_rate(uint32_t in_rate, uint32_t out_rate, uint64_t n_in, uint64_t *n_out, uint32_t *mode, uint32_t *p,
              uint32_t *q, std::shared_ptr<FracTable> *table)
{
    if (in_rate == 0 || out_rate == 0) return fail(AF_ERR_INVALID, "sample rate must be positive");
    RsRecurrence probe;
    probe.init(in_rate, out_rate);
    *mode = probe.mode(); *p = probe.p; *q = probe.q;
    if (probe.passthrough) { *n_out = n_in; return AF_OK; }
    if (probe.end_idx <= 0)
        return fail(AF_ERR_RESAMPLING_FAILED, "unsupported resampling ratio %u -> %u (step %.3f exceeds the 128-frame chunk)",
                    in_rate, out_rate, probe.t);
    const uint64_t chunks = (n_in + RS_CHUNK - 1) / RS_CHUNK;
    if (probe.exact) { *n_out = rs_exact_count(probe, chunks); return AF_OK; }
    std::lock_guard<std::mutex> lk(cur_ctx().mu);
    RatePlan &pl = cur_ctx().plans[((uint64_t)in_rate << 32) | out_rate];
    if (pl.rec.in_rate == 0) pl.rec.init(in_rate, out_rate);
    bool grew = false;
    while (pl.cum.size() - 1 < chunks) {
        pl.rec.step(&pl.frac);
        pl.cum.push_back(pl.rec.n_out);
        grew = true;
    }
    *n_out = pl.cum[chunks];
    if (table) {
        if (grew || !pl.dev || pl.dev->n < pl.frac.size()) {
            auto t = std::make_shared<FracTable>();
            t->n = pl.frac.size();
            if (t->n) {
                // Device form of the table: the fraction the reference's f64 recurrence produces, with the SIGN BIT set where
                // the recurrence sits just below an exactly integer position (frac ~ 1 and floor one less than the exact
                // integer arithmetic of the kernel gives): the kernel then needs no float round trip to find the tap --
                // k -= sign, frac = |entry|.  (Fractions are never negative, and a flagged one is never 0.)
                std::vector<float> enc(pl.frac);
                for (size_t n = 0; n < enc.size(); ++n) {
                    long long k; uint32_t rem;
                    resample_pos(n, pl.rec.p, pl.rec.q, &k, &rem);
                    if (rem == 0 && enc[n] >= 0.5f) enc[n] = -enc[n];
                }
                // (16 floats of slack: the kernel fetches whole quads)
                AF_CUDA(t->d.alloc(t->n + 16));
                AF_CUDA(cudaMemset(t->d.get(), 0, (t->n + 16) * sizeof(float)));
                AF_CUDA(cudaMemcpy(t->d.get(), enc.data(), t->n * sizeof(float), cudaMemcpyHostToDevice));
            }
            pl.dev = t;
        }
        *table = pl.dev;
    }
    return AF_OK;
}

}  // namespace

// ------------------------------------------------------------------------------------------
// library
// ------------------------------------------------------------------------------------------
extern "C" {

AF_API const char *af_version(void) { return "audioflow-b200 0.1.0 (sm_100a)"; }

AF_API size_t af_last_error(char *buf, size_t cap)
{
    if (buf && cap) {
        size_t n = g_err.size() < cap - 1 ? g_err.size() : cap - 1;
        memcpy(buf, g_err.data(), n);
        buf[n] = 0;
    }
    return g_err.size();
}

AF_API int af_device_count(int *count)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) { (void)cudaGetLastError(); n = 0; }
    if (count) *count = n;
    return AF_OK;
}

AF_API uint64_t af_kernel_launch_count(void) { return g_launches.load(); }

AF_API int af_debug_pipe_stats(uint64_t out[32])
{
    if (!out) return fail(AF_ERR_INVALID, "null output");
    unsigned long long tmp[32];
    AF_CUDA(cudaDeviceSynchronize());
    AF_CUDA(fused_pipe_stats(tmp));
    for (int i = 0; i < 32; ++i) out[i] = tmp[i];
    return AF_OK;
}

AF_API int af_debug_live_allocations(uint64_t *device, uint64_t *pinned)
{
    if (device) *device = g_live_allocs[(int)Mem::Device].load();
    if (pinned) *pinned = g_live_allocs[(int)Mem::Pinned].load();
    return AF_OK;
}

AF_API int af_init(int device)
{
    // selects `device` for the calling thread (initialising it on first use); device < 0: keep the thread's / the
    // process default, or take the thread's current CUDA device when nothing is initialised yet
    if (device < 0) return require_ctx();
    int rc = init_device(device);
    if (rc != AF_OK) return rc;
    t_dev = device;
    AF_CUDA(cudaSetDevice(device));
    return AF_OK;
}

AF_API int af_current_device(void) { return t_dev >= 0 ? t_dev : g_default_dev.load(); }

AF_API int af_set_stream(void *cuda_stream)
{
    int rc = require_ctx();
    if (rc) return rc;
    Context &c = cur_ctx();
    c.stream = cuda_stream ? (cudaStream_t)cuda_stream : c.own;
    return AF_OK;
}

AF_API int af_shutdown(void)
{
    comm_shutdown_all();
    std::lock_guard<std::mutex> lk(g_init_mu);
    int prev = 0;
    (void)cudaGetDevice(&prev);
    for (int d = 0; d < MAX_DEV; ++d) {
        Context &c = g_ctxs[d];
        if (!c.ready) continue;
        (void)cudaSetDevice(d);
        cudaDeviceSynchronize();
        c.plans.clear();
        c.scratch_in.reset(); c.scratch_out.reset(); c.scratch_aux.reset(); c.scratch_jobs.reset();
        c.d_fft.reset();
        if (c.own) cudaStreamDestroy(c.own);
        if (c.side) cudaStreamDestroy(c.side);
        c.stream = nullptr; c.own = nullptr; c.side = nullptr;
        c.ready = false;
        c.device = -1;
    }
    (void)cudaSetDevice(prev);
    g_default_dev.store(-1);
    t_dev = -1;
    return AF_OK;
}

AF_API int af_host_alloc(void **ptr, size_t bytes)
{
    if (!ptr) return fail(AF_ERR_INVALID, "null pointer");
    int rc = require_ctx();
    if (rc) return rc;
    PinnedBuf<uint8_t> b;
    AF_CUDA(b.alloc(bytes ? bytes : 1, cudaHostAllocPortable));    // pinned for every device of the process
    *ptr = b.release();
    return AF_OK;
}

AF_API int af_host_free(void *ptr)
{
    AF_CUDA(PinnedBuf<uint8_t>::adopt(static_cast<uint8_t *>(ptr)).reset());
    return AF_OK;
}

AF_API int af_set_kernel_variant(const char *name)
{
    if (!name) return fail(AF_ERR_INVALID, "null variant name");
    std::string v(name);
    if (v != "auto" && v != "sync" && v != "tma") return fail(AF_ERR_INVALID, "unknown kernel variant '%s'", name);
    g_variant = v;
    return AF_OK;
}

// ------------------------------------------------------------------------------------------
// AudioFrame::to_mono (capture.rs:30-42)
// ------------------------------------------------------------------------------------------
AF_API int af_to_mono(const float *samples, size_t n_samples, uint16_t channels, float *out, size_t out_cap,
                      size_t *n_out)
{
    if (channels == 0) return fail(AF_ERR_INVALID, "channels must be >= 1");
    if ((!samples || !out) && n_samples) return fail(AF_ERR_INVALID, "null buffer");
    int rc = require_ctx();
    if (rc) return rc;
    const size_t frames = (n_samples + channels - 1) / channels;
    if (out_cap < frames) return fail(AF_ERR_CAPACITY, "output capacity %zu < %zu frames", out_cap, frames);
    if (n_out) *n_out = frames;
    if (frames == 0) return AF_OK;
    std::lock_guard<std::mutex> lk(cur_ctx().mu);
    AF_CUDA(reserve(cur_ctx().scratch_in, n_samples * sizeof(float)));
    AF_CUDA(reserve(cur_ctx().scratch_out, frames * sizeof(float)));
    cudaStream_t st = cur_ctx().stream;
    AF_CUDA(cudaMemcpyAsync(cur_ctx().scratch_in.get(), samples, n_samples * sizeof(float), cudaMemcpyHostToDevice, st));
    AF_CUDA(launch_to_mono((const float *)cur_ctx().scratch_in.get(), n_samples, channels, (float *)cur_ctx().scratch_out.get(), frames, st));
    count_launch();
    AF_CUDA(cudaMemcpyAsync(out, cur_ctx().scratch_out.get(), frames * sizeof(float), cudaMemcpyDeviceToHost, st));
    AF_CUDA(cudaStreamSynchronize(st));
    return AF_OK;
}

// ------------------------------------------------------------------------------------------
// AudioResampler / BatchResampler (resampler.rs)
// ------------------------------------------------------------------------------------------
struct af_resampler {
    int device = -1;                  // the GPU the object was created on
    RsRecurrence rec;
    float hist[2 * RS_POLY];          // the last 16 input frames (rubato's buffer head)
    std::vector<float> frac;          // scratch
    std::vector<float> stage;         // scratch: hist + chunks
};

static int resampler_run_chunks(af_resampler *r, const float *input, size_t n_chunks, float *out, size_t out_cap,
                                size_t *n_out)
{
    // runs n_chunks complete 128-frame chunks through the GPU; input has n_chunks * 128 frames
    AF_SCOPE(r->device);
    const uint64_t c0 = r->rec.chunks;
    const uint64_t n_begin = r->rec.n_out;
    RsRecurrence saved = r->rec;
    r->frac.clear();
    for (size_t c = 0; c < n_chunks; ++c) r->rec.step(r->rec.exact ? nullptr : &r->frac);
    const uint64_t n_end = r->rec.n_out;
    const size_t produced = (size_t)(n_end - n_begin);
    if (produced > out_cap) {
        r->rec = saved;
        return fail(AF_ERR_CAPACITY, "output capacity %zu < %zu produced frames", out_cap, produced);
    }
    const size_t n_in = n_chunks * RS_CHUNK;
    r->stage.resize(2 * RS_POLY + n_in);
    memcpy(r->stage.data(), r->hist, sizeof(r->hist));
    memcpy(r->stage.data() + 2 * RS_POLY, input, n_in * sizeof(float));

    std::lock_guard<std::mutex> lk(cur_ctx().mu);
    cudaStream_t st = cur_ctx().stream;
    const size_t in_bytes = r->stage.size() * sizeof(float);
    const size_t frac_bytes = r->frac.size() * sizeof(float);
    AF_CUDA(reserve(cur_ctx().scratch_in, in_bytes));
    AF_CUDA(reserve(cur_ctx().scratch_aux, frac_bytes + 16));
    AF_CUDA(reserve(cur_ctx().scratch_out, produced * sizeof(float) + 16));
    AF_CUDA(reserve(cur_ctx().scratch_jobs, sizeof(ResampleJob)));
    AF_CUDA(cudaMemcpyAsync(cur_ctx().scratch_in.get(), r->stage.data(), in_bytes, cudaMemcpyHostToDevice, st));
    if (frac_bytes) AF_CUDA(cudaMemcpyAsync(cur_ctx().scratch_aux.get(), r->frac.data(), frac_bytes, cudaMemcpyHostToDevice, st));
    ResampleJob job;
    job.data = (const float *)cur_ctx().scratch_in.get();
    job.data_base = (long long)(c0 * RS_CHUNK) - 2 * RS_POLY;
    job.n_valid_end = (long long)((c0 + n_chunks) * RS_CHUNK);
    job.n_begin = n_begin; job.n_end = n_end;
    job.p = r->rec.p; job.q = r->rec.q; job.mode = r->rec.mode();
    job.frac = (const float *)cur_ctx().scratch_aux.get() - n_begin;      // indexed by the global output index
    job.out = (float *)cur_ctx().scratch_out.get();
    AF_CUDA(cudaMemcpyAsync(cur_ctx().scratch_jobs.get(), &job, sizeof(job), cudaMemcpyHostToDevice, st));
    if (produced) {
        AF_CUDA(launch_resample_jobs((const ResampleJob *)cur_ctx().scratch_jobs.get(), 1, (uint32_t)produced, st));
        count_launch();
        AF_CUDA(cudaMemcpyAsync(out, cur_ctx().scratch_out.get(), produced * sizeof(float), cudaMemcpyDeviceToHost, st));
    }
    AF_CUDA(cudaStreamSynchronize(st));
    memcpy(r->hist, r->stage.data() + r->stage.size() - 2 * RS_POLY, sizeof(r->hist));
    *n_out = produced;
    return AF_OK;
}

AF_API int af_resampler_create(uint32_t input_rate, uint32_t output_rate, af_resampler **out)
{
    if (!out) return fail(AF_ERR_INVALID, "null out pointer");
    if (input_rate == 0 || output_rate == 0) return fail(AF_ERR_RESAMPLING_FAILED, "sample rates must be positive");
    int rc = require_ctx();
    if (rc) return rc;
    af_resampler *r = new af_resampler;
    r->device = cur_device();
    r->rec.init(input_rate, output_rate);
    memset(r->hist, 0, sizeof(r->hist));
    if (!r->rec.passthrough && r->rec.end_idx <= 0) {
        delete r;
        return fail(AF_ERR_RESAMPLING_FAILED, "unsupported resampling ratio %u -> %u", input_rate, output_rate);
    }
    *out = r;
    return AF_OK;
}

AF_API void af_resampler_destroy(af_resampler *r) { delete r; }
AF_API uint32_t af_resampler_input_rate(const af_resampler *r) { return r ? r->rec.in_rate : 0; }
AF_API uint32_t af_resampler_output_rate(const af_resampler *r) { return r ? r->rec.out_rate : 0; }
AF_API int af_resampler_needs_resampling(const af_resampler *r) { return r && r->rec.in_rate != r->rec.out_rate; }
AF_API size_t af_resampler_chunk_size(const af_resampler *r) { return (r && !r->rec.passthrough) ? RS_CHUNK : 0; }

AF_API int af_resampler_process(af_resampler *r, const float *input, size_t n, float *out, size_t out_cap, size_t *n_out)
{
    if (!r || !n_out || ((!input || !out) && n)) return fail(AF_ERR_INVALID, "null argument");
    if (r->rec.passthrough) {                         // resampler.rs:72-75: Ok(input.to_vec())
        if (out_cap < n) return fail(AF_ERR_CAPACITY, "output capacity %zu < %zu", out_cap, n);
        memcpy(out, input, n * sizeof(float));
        *n_out = n;
        return AF_OK;
    }
    if (n < RS_CHUNK)                                 // rubato ResampleError::InsufficientInputBufferSize
        return fail(AF_ERR_RESAMPLING_FAILED, "Insufficient buffer size %zu for input channel 0, expected %d", n, RS_CHUNK);
    return resampler_run_chunks(r, input, 1, out, out_cap, n_out);
}

AF_API size_t af_resample_max_output(uint32_t input_rate, uint32_t output_rate, size_t n_in)
{
    if (input_rate == output_rate || input_rate == 0) return n_in;
    const size_t chunks = (n_in + RS_CHUNK - 1) / RS_CHUNK;
    const double per = (double)RS_CHUNK * (double)output_rate / (double)input_rate;
    return (size_t)((double)chunks * per) + chunks + 64;
}

AF_API int af_resample_output_len(uint32_t input_rate, uint32_t output_rate, size_t n_in, size_t *n_out)
{
    if (!n_out) return fail(AF_ERR_INVALID, "null out pointer");
    uint64_t n = 0; uint32_t mode, p, q;
    int rc = plan_rate(input_rate, output_rate, n_in, &n, &mode, &p, &q, nullptr);
    if (rc) return rc;
    *n_out = (size_t)n;
    return AF_OK;
}

struct af_batch_resampler {
    af_resampler rs;
    std::vector<float> buffer;        // BatchResampler::buffer (resampler.rs:118): always < 128 frames after process
};

AF_API int af_batch_resampler_create(uint32_t input_rate, uint32_t output_rate, af_batch_resampler **out)
{
    if (!out) return fail(AF_ERR_INVALID, "null out pointer");
    af_resampler *r = nullptr;
    int rc = af_resampler_create(input_rate, output_rate, &r);
    if (rc) return rc;
    af_batch_resampler *b = new af_batch_resampler;
    b->rs = *r;
    delete r;
    *out = b;
    return AF_OK;
}
AF_API void af_batch_resampler_destroy(af_batch_resampler *b) { delete b; }

AF_API int af_batch_resampler_process(af_batch_resampler *b, const float *input, size_t n, float *out, size_t out_cap,
                                      size_t *n_out)
{
    if (!b || !n_out || ((!input || !out) && n)) return fail(AF_ERR_INVALID, "null argument");
    *n_out = 0;
    if (b->rs.rec.passthrough) {                      // documented deviation: the reference never returns here
        if (out_cap < n) return fail(AF_ERR_CAPACITY, "output capacity %zu < %zu", out_cap, n);
        memcpy(out, input, n * sizeof(float));
        *n_out = n;
        return AF_OK;
    }
    b->buffer.insert(b->buffer.end(), input, input + n);
    const size_t chunks = b->buffer.size() / RS_CHUNK;
    if (chunks == 0) return AF_OK;
    int rc = resampler_run_chunks(&b->rs, b->buffer.data(), chunks, out, out_cap, n_out);
    if (rc) { b->buffer.resize(b->buffer.size() - n); return rc; }
    b->buffer.erase(b->buffer.begin(), b->buffer.begin() + chunks * RS_CHUNK);
    return AF_OK;
}

AF_API int af_batch_resampler_flush(af_batch_resampler *b, float *out, size_t out_cap, size_t *n_out)
{
    if (!b || !n_out) return fail(AF_ERR_INVALID, "null argument");
    *n_out = 0;
    if (b->buffer.empty()) return AF_OK;
    if (b->rs.rec.passthrough) { b->buffer.clear(); return AF_OK; }
    std::vector<float> chunk(RS_CHUNK, 0.0f);         // resampler.rs:156-157: resize(chunk_size, 0.0)
    memcpy(chunk.data(), b->buffer.data(), b->buffer.size() * sizeof(float));
    int rc = resampler_run_chunks(&b->rs, chunk.data(), 1, out, out_cap, n_out);
    if (rc) return rc;
    b->buffer.clear();
    return AF_OK;
}

// ------------------------------------------------------------------------------------------
// VoiceActivityDetector (vad.rs)
// ------------------------------------------------------------------------------------------
struct af_vad {
    int device = -1;                  // the GPU the detector state lives on
    af_vad_config cfg;
    VadParams prm;
    VadState host;                    // mirror of the device state after the last call
    DevBuf<VadState> dev;
};

static VadParams make_vad_params(const af_vad_config &c)
{
    VadParams p;
    p.alpha = c.smoothing_factor;
    p.e_min = vad_energy_threshold(c.threshold_db);
    p.silence_timeout = c.silence_timeout_frames;
    p.min_speech = c.min_speech_frames;
    return p;
}

// the scan records of n configurations: the e_min bisection (vad_energy_threshold) runs once per distinct threshold
static void make_scan_recs(const af_vad_config *cfgs, size_t n, ScanRec *out)
{
    std::map<uint32_t, float> e_min;                  // threshold bits -> e_min
    for (size_t i = 0; i < n; ++i) {
        uint32_t bits;
        memcpy(&bits, &cfgs[i].threshold_db, sizeof(bits));
        auto it = e_min.find(bits);
        if (it == e_min.end()) it = e_min.emplace(bits, vad_energy_threshold(cfgs[i].threshold_db)).first;
        VadParams p;
        p.alpha = cfgs[i].smoothing_factor;
        p.e_min = it->second;
        p.silence_timeout = cfgs[i].silence_timeout_frames;
        p.min_speech = cfgs[i].min_speech_frames;
        out[i] = scan_rec(p);
    }
}

static bool same_rec(const ScanRec &a, const ScanRec &b) { return memcmp(&a, &b, sizeof(ScanRec)) == 0; }
static_assert(sizeof(ScanRec) == 32, "ScanRec has no padding: same_rec compares bytes");

AF_API void af_vad_config_default(af_vad_config *cfg)
{
    if (!cfg) return;
    cfg->threshold_db = -50.0f;
    cfg->smoothing_factor = 0.3f;
    cfg->silence_timeout_frames = 15;
    cfg->min_speech_frames = 3;
}

AF_API int af_vad_create(const af_vad_config *cfg, af_vad **out)
{
    if (!out) return fail(AF_ERR_INVALID, "null out pointer");
    int rc = require_ctx();
    if (rc) return rc;
    af_vad *v = new af_vad;
    v->device = cur_device();
    if (cfg) v->cfg = *cfg; else af_vad_config_default(&v->cfg);
    v->prm = make_vad_params(v->cfg);
    memset(&v->host, 0, sizeof(v->host));
    cudaError_t e = v->dev.alloc(1);
    if (e == cudaSuccess) e = cudaMemset(v->dev.get(), 0, sizeof(VadState));
    if (e != cudaSuccess) { delete v; AF_CUDA(e); }
    *out = v;
    return AF_OK;
}

AF_API void af_vad_destroy(af_vad *v)
{
    if (!v) return;
    DevScope scope_(v->device);
    delete v;
}

AF_API int af_vad_detect_frames(af_vad *v, const float *samples, size_t n, uint32_t frame_len, uint32_t hop,
                                uint8_t *states, size_t states_cap, size_t *n_frames)
{
    if (!v || (!samples && n)) return fail(AF_ERR_INVALID, "null argument");
    if (hop == 0) return fail(AF_ERR_INVALID, "hop must be positive");
    size_t T = n >= frame_len ? 1 + (n - frame_len) / hop : 0;
    if (frame_len == 0) T = 0;
    if (n_frames) *n_frames = T;
    if (T == 0) return AF_OK;
    if (states && states_cap < T) return fail(AF_ERR_CAPACITY, "states capacity %zu < %zu frames", states_cap, T);
    AF_SCOPE(v->device);
    std::lock_guard<std::mutex> lk(cur_ctx().mu);
    cudaStream_t st = cur_ctx().stream;
    AF_CUDA(reserve(cur_ctx().scratch_in, n * sizeof(float)));
    AF_CUDA(reserve(cur_ctx().scratch_aux, T * sizeof(float)));
    AF_CUDA(reserve(cur_ctx().scratch_out, T));
    AF_CUDA(cudaMemcpyAsync(cur_ctx().scratch_in.get(), samples, n * sizeof(float), cudaMemcpyHostToDevice, st));
    EnergyJob ej{};
    ej.y = (const float *)cur_ctx().scratch_in.get(); ej.y_stride = 0; ej.n_frames = nullptr; ej.n_frames_all = (uint32_t)T;
    ej.frame_len = frame_len; ej.hop = hop; ej.energy = (float *)cur_ctx().scratch_aux.get(); ej.energy_stride = 0; ej.n_streams = 1;
    AF_CUDA(launch_frame_energy(ej, st));
    ScanJob sj{};
    sj.energy = (const float *)cur_ctx().scratch_aux.get(); sj.energy_stride = 0; sj.n_frames = nullptr; sj.n_frames_all = (uint32_t)T;
    sj.states = (uint8_t *)cur_ctx().scratch_out.get(); sj.states_stride = 0; sj.state_io = v->dev.get(); sj.final_out = nullptr;
    sj.prm = v->prm; sj.n_streams = 1;
    AF_CUDA(launch_vad_scan(sj, st));
    count_launch(2);
    if (states) AF_CUDA(cudaMemcpyAsync(states, cur_ctx().scratch_out.get(), T, cudaMemcpyDeviceToHost, st));
    AF_CUDA(cudaMemcpyAsync(&v->host, v->dev.get(), sizeof(VadState), cudaMemcpyDeviceToHost, st));
    AF_CUDA(cudaStreamSynchronize(st));
    return AF_OK;
}

AF_API int af_vad_detect(af_vad *v, const float *frame, size_t n, uint8_t *state)
{
    if (!v) return fail(AF_ERR_INVALID, "null detector");
    if (n == 0) {
        // calculate_energy returns 0.0 for an empty frame (vad.rs:158-160) and the state machine still steps:
        // feed one zero sample, whose mean square is exactly 0.0 as well
        const float zero = 0.0f;
        uint8_t s = 0;
        int rc = af_vad_detect_frames(v, &zero, 1, 1, 1, &s, 1, nullptr);
        if (state) *state = s;
        return rc;
    }
    if (n > 0xffffffffull) return fail(AF_ERR_INVALID, "frame too long");
    uint8_t s = 0;
    int rc = af_vad_detect_frames(v, frame, n, (uint32_t)n, (uint32_t)n, &s, 1, nullptr);
    if (state) *state = s;
    return rc;
}

AF_API int af_vad_reset(af_vad *v)
{
    if (!v) return fail(AF_ERR_INVALID, "null detector");
    memset(&v->host, 0, sizeof(v->host));
    AF_SCOPE(v->device);
    AF_CUDA(cudaMemset(v->dev.get(), 0, sizeof(VadState)));
    return AF_OK;
}
AF_API int af_vad_state(const af_vad *v) { return v ? v->host.state : 0; }
AF_API float af_vad_energy_db(const af_vad *v)
{
    // energy_to_dbfs(smoothed_energy) (vad.rs:171-176,192-194); host libm, same as the threshold derivation
    if (!v || !(v->host.smoothed > 0.0f)) return -INFINITY;
    return 20.0f * log10f(v->host.smoothed);
}
AF_API int af_vad_is_speaking(const af_vad *v) { return v && v->host.state == AF_VAD_SPEECH; }
AF_API uint64_t af_vad_speech_frame_count(const af_vad *v) { return v ? v->host.speech_frames : 0; }
AF_API float af_vad_smoothed_energy(const af_vad *v) { return v ? v->host.smoothed : 0.0f; }

AF_API int af_vad_frame_energy(const float *frame, size_t n, float *energy)
{
    if (!energy || (!frame && n)) return fail(AF_ERR_INVALID, "null argument");
    int rc = require_ctx();
    if (rc) return rc;
    if (n == 0) { *energy = 0.0f; return AF_OK; }
    std::lock_guard<std::mutex> lk(cur_ctx().mu);
    cudaStream_t st = cur_ctx().stream;
    AF_CUDA(reserve(cur_ctx().scratch_in, n * sizeof(float)));
    AF_CUDA(reserve(cur_ctx().scratch_aux, sizeof(float)));
    AF_CUDA(cudaMemcpyAsync(cur_ctx().scratch_in.get(), frame, n * sizeof(float), cudaMemcpyHostToDevice, st));
    EnergyJob ej{};
    ej.y = (const float *)cur_ctx().scratch_in.get(); ej.n_frames_all = 1; ej.frame_len = (uint32_t)n; ej.hop = (uint32_t)n;
    ej.energy = (float *)cur_ctx().scratch_aux.get(); ej.n_streams = 1;
    AF_CUDA(launch_frame_energy(ej, st));
    count_launch();
    AF_CUDA(cudaMemcpyAsync(energy, cur_ctx().scratch_aux.get(), sizeof(float), cudaMemcpyDeviceToHost, st));
    AF_CUDA(cudaStreamSynchronize(st));
    return AF_OK;
}

AF_API int af_pcm16_encode(const float *samples, size_t n, int16_t *out)
{
    if ((!samples || !out) && n) return fail(AF_ERR_INVALID, "null buffer");
    int rc = require_ctx();
    if (rc) return rc;
    if (n == 0) return AF_OK;
    std::lock_guard<std::mutex> lk(cur_ctx().mu);
    cudaStream_t st = cur_ctx().stream;
    AF_CUDA(reserve(cur_ctx().scratch_in, n * sizeof(float)));
    AF_CUDA(reserve(cur_ctx().scratch_out, n * sizeof(int16_t)));
    AF_CUDA(cudaMemcpyAsync(cur_ctx().scratch_in.get(), samples, n * sizeof(float), cudaMemcpyHostToDevice, st));
    AF_CUDA(launch_pcm16((const float *)cur_ctx().scratch_in.get(), n, (int16_t *)cur_ctx().scratch_out.get(), st));
    count_launch();
    AF_CUDA(cudaMemcpyAsync(out, cur_ctx().scratch_out.get(), n * sizeof(int16_t), cudaMemcpyDeviceToHost, st));
    AF_CUDA(cudaStreamSynchronize(st));
    return AF_OK;
}

AF_API size_t af_pcm16_base64_len(size_t n_samples) { return 4 * ((2 * n_samples + 2) / 3); }

AF_API int af_pcm16_base64(const float *samples, size_t n, char *out, size_t out_cap, size_t *n_out)
{
    if (n_out) *n_out = 0;
    if ((!samples || !out) && n) return fail(AF_ERR_INVALID, "null buffer");
    const size_t need = af_pcm16_base64_len(n);
    if (out_cap < need) return fail(AF_ERR_CAPACITY, "base64 output needs %zu characters, capacity %zu", need, out_cap);
    int rc = require_ctx();
    if (rc) return rc;
    if (n == 0) return AF_OK;
    std::lock_guard<std::mutex> lk(cur_ctx().mu);
    cudaStream_t st = cur_ctx().stream;
    AF_CUDA(reserve(cur_ctx().scratch_in, n * sizeof(float)));
    AF_CUDA(reserve(cur_ctx().scratch_out, need));
    AF_CUDA(cudaMemcpyAsync(cur_ctx().scratch_in.get(), samples, n * sizeof(float), cudaMemcpyHostToDevice, st));
    AF_CUDA(launch_pcm16_base64((const float *)cur_ctx().scratch_in.get(), n, (char *)cur_ctx().scratch_out.get(), st));
    count_launch();
    AF_CUDA(cudaMemcpyAsync(out, cur_ctx().scratch_out.get(), need, cudaMemcpyDeviceToHost, st));
    AF_CUDA(cudaStreamSynchronize(st));
    if (n_out) *n_out = need;
    return AF_OK;
}

AF_API int af_vad_segments(const uint8_t *states, uint64_t vad_stride, const uint32_t *n_frames, size_t n_streams,
                           uint32_t *seg, uint32_t seg_cap, uint32_t *n_seg, void *cuda_stream)
{
    if (!states || !n_frames || !seg || !n_seg) return fail(AF_ERR_INVALID, "null argument");
    int rc = require_ctx();
    if (rc) return rc;
    const int owner = device_of_pointer(states);                 // the GPU that holds the states (else the thread's device)
    AF_SCOPE(owner >= 0 && device_ctx(owner) ? owner : cur_device());
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : cur_ctx().stream;
    AF_CUDA(launch_vad_segments(states, vad_stride, n_frames, (uint32_t)n_streams, seg, seg_cap, n_seg, st));
    count_launch();
    if (!cuda_stream) AF_CUDA(cudaStreamSynchronize(st));
    return AF_OK;
}

AF_API int af_vad_segments_preroll(uint32_t *seg, uint32_t seg_cap, const uint32_t *n_seg, size_t n_streams,
                                   uint32_t preroll_frames, void *cuda_stream)
{
    if (!seg || !n_seg) return fail(AF_ERR_INVALID, "null argument");
    if (preroll_frames == 0) return AF_OK;                       // the segments as they are
    int rc = require_ctx();
    if (rc) return rc;
    const int owner = device_of_pointer(seg);
    AF_SCOPE(owner >= 0 && device_ctx(owner) ? owner : cur_device());
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : cur_ctx().stream;
    AF_CUDA(launch_vad_segments_preroll(seg, seg_cap, n_seg, (uint32_t)n_streams, preroll_frames, st));
    if ((uint64_t)n_streams * seg_cap) count_launch();
    if (!cuda_stream) AF_CUDA(cudaStreamSynchronize(st));
    return AF_OK;
}

AF_API int af_vad_gate(const float *pcm, uint64_t pcm_stride, const float *logmel, uint64_t logmel_stride, uint32_t n_mels,
                       const uint32_t *n_out, uint32_t hop, const uint32_t *seg, uint32_t seg_cap, const uint32_t *n_seg,
                       size_t n_streams, const af_gate_outputs *out, void *cuda_stream)
{
    if (!seg || !n_seg || !out || !out->seg_offset || !out->n_frames) return fail(AF_ERR_INVALID, "null argument");
    if (hop == 0) return fail(AF_ERR_INVALID, "hop must be positive");
    if ((out->pcm && !pcm) || (out->logmel && (!logmel || n_mels == 0))) return fail(AF_ERR_INVALID, "gated output requested without its source");
    int rc = require_ctx();
    if (rc) return rc;
    const int owner = device_of_pointer(seg);
    AF_SCOPE(owner >= 0 && device_ctx(owner) ? owner : cur_device());
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : cur_ctx().stream;
    GateJob J{};
    J.pcm = out->pcm ? pcm : nullptr; J.pcm_stride = pcm_stride;
    J.logmel = out->logmel ? logmel : nullptr; J.logmel_stride = logmel_stride;
    J.n_mels = n_mels; J.hop = hop; J.n_out = n_out;
    J.seg = seg; J.seg_cap = seg_cap; J.n_seg = n_seg;
    J.off = out->seg_offset; J.total = out->n_frames;
    J.out_pcm = out->pcm; J.out_pcm_stride = out->pcm_stride;
    J.out_lm = out->logmel; J.out_lm_stride = out->logmel_stride;
    J.n_streams = (uint32_t)n_streams;
    AF_CUDA(launch_vad_gate(J, st));
    count_launch((J.out_pcm || J.out_lm) ? 2 : 1);
    if (!cuda_stream) AF_CUDA(cudaStreamSynchronize(st));
    return AF_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------
// batched pipeline
// ------------------------------------------------------------------------------------------
struct af_pipeline {
    af_pipeline_config cfg;
    VadParams vad_prm;
    MelTables h_mel;                              // built once on the host ...
    DevBuf<MelTables> d_mel[MAX_DEV];             // ... and copied to every device that runs the pipeline, on first use
    std::mutex mu;
};

namespace {
// the pipeline's mel tables on the calling thread's device (nullptr without features or on a CUDA failure)
MelTables *pipe_mel(af_pipeline *p)
{
    if (!p->cfg.n_mels) return nullptr;
    const int dev = cur_device();
    std::lock_guard<std::mutex> lk(p->mu);
    if (!p->d_mel[dev].get()) {
        cudaError_t e = p->d_mel[dev].alloc(1);
        if (e == cudaSuccess) e = cudaMemcpy(p->d_mel[dev].get(), &p->h_mel, sizeof(MelTables), cudaMemcpyHostToDevice);
        if (e != cudaSuccess) {
            p->d_mel[dev].reset();
            fail(AF_ERR_CUDA, "mel tables: %s", cudaGetErrorString(e));
        }
    }
    return p->d_mel[dev].get();
}
}  // namespace

namespace {

struct HostStream {                   // planned stream (host side)
    af_stream_desc desc;
    uint32_t n_in, n_out, n_frames, n_vad_frames, mode, p, q;
    std::shared_ptr<FracTable> table;
};

struct SubBatch {                     // a group of streams resident on the device together
    size_t first = 0, count = 0;      // range in af_batch::streams
    std::vector<StreamDev> h_streams;
    std::vector<TileDev> h_tiles;
    DevBuf<StreamDev> d_streams;
    DevBuf<TileDev> d_tiles;
    DevBuf<uint32_t> d_nframes, d_nvad;
    std::vector<size_t> in_off;       // host mode: byte offset of each stream inside the slot input buffer
    size_t in_bytes = 0;
    DevBuf<uint32_t> d_scan;          // long streams: scratch of the many-CTA VAD scan (launch_vad_scan)
    DevBuf<ScanRec> d_recs;           // its streams' VAD records (af_batch_set_vad_configs), or empty: the pipeline's
    uint32_t n_seq = 0;               // records of d_recs flagged for the sequential scan kernel
    bool quarters = false;            // some stream stages its input in quarter steps (f32 stereo)
    bool split = false;               // some stream is not 48 kHz mono f32 -> 16 kHz (FusedParams::split)
    uint32_t per_p = 0, per_q = 0;    // p / q of the batch's RS_TABLE streams when the output period fits the kernel's position table
    bool no_merge = false;            // host mode: a merged copy was refused (rows adjacent in memory but separately allocated)
};

// af_batch_set_resampler(AF_RESAMPLE_POLYPHASE): the FIR writes each sub-batch's 16 kHz rows into a scratch block and
// the fused kernel runs over them as 16 kHz mono f32 streams (counts, frames and strides are the batch's own)
struct Polyphase {
    std::vector<HostStream> rows;             // stream i as the fused kernel sees it: 16 kHz mono f32, n_in = n_out
    std::map<uint32_t, DevBuf<float>> taps;   // one tap table per input rate of the batch
    std::vector<DevBuf<float>> d_rows;        // the rows: one block (device batches) or one per slot (host batches)
    std::vector<SubBatch> subs;               // the fused plan of each sub-batch over its rows
    std::vector<FirJob> jobs;                 // the FIR launch of each sub-batch
    std::vector<DevBuf<FirStream>> d_fir;
    std::vector<DevBuf<uint2>> d_tiles;
};

}  // namespace

struct af_batch {
    af_pipeline *pipe = nullptr;
    int device = -1;                  // the GPU the batch was planned for
    MelTables *d_mel = nullptr;       // the pipeline's mel tables on that GPU
    int mem = AF_MEM_DEVICE;
    std::vector<HostStream> streams;
    std::vector<SubBatch> subs;
    uint64_t max_out = 0, max_frames = 0, max_vad = 0;
    uint64_t pcm_stride = 0, logmel_stride = 0, vad_stride = 0;
    // device scratch for outputs the caller did not ask for but the pipeline needs
    DevBuf<float> d_energy; uint64_t energy_stride = 0;
    DevBuf<float> d_pcm_scratch;
    // host mode slots
    struct Slot {
        DevBuf<char> d_in; DevBuf<float> d_pcm; DevBuf<int16_t> d_pcm16; DevBuf<float> d_logmel; DevBuf<uint8_t> d_vad;
        DevBuf<float> d_energy; DevBuf<VadState> d_final;
        cudaStream_t st = nullptr;
    };
    std::vector<Slot> slots;
    size_t slot_rows = 0;
    std::unique_ptr<Polyphase> poly;  // polyphase resampling (af_batch_set_resampler), or null: the cubic path
};

namespace {

int build_sub(const std::vector<HostStream> &streams, SubBatch &sb, const void *slot_in_base)
{
    // (re)build the device tables of a sub-batch; slot_in_base != null (host mode, polyphase rows) rebases the inputs
    sb.h_streams.resize(sb.count);
    sb.h_tiles.clear();
    sb.quarters = false;
    sb.per_p = sb.per_q = 0;
    sb.split = false;
    std::vector<uint32_t> nf(sb.count), nv(sb.count);
    for (size_t i = 0; i < sb.count; ++i) {
        const HostStream &hs = streams[sb.first + i];
        StreamDev &d = sb.h_streams[i];
        memset(&d, 0, sizeof(d));
        d.data = slot_in_base ? (const void *)((const char *)slot_in_base + sb.in_off[i]) : hs.desc.data;
        d.n_samples = hs.desc.n_samples;
        d.n_in = hs.n_in; d.n_out = hs.n_out; d.n_frames = hs.n_frames; d.n_vad_frames = hs.n_vad_frames;
        d.channels = hs.desc.channels; d.format = hs.desc.format;
        d.p = hs.p; d.q = hs.q; d.mode = hs.mode;
        d.frac = hs.table ? hs.table->d.get() : nullptr;
        {   // does the raw input of one step fit the shared-memory stage of the fused kernel?
            const uint64_t bps = hs.desc.format == AF_FMT_I16 ? 2 : 4;
            // (a step is staged in two fills of half a step each, or in four of a quarter: whichever fits a stage buffer)
            d.staged = 0;
            for (int parts = 2; parts <= MAX_PARTS && !d.staged; parts += 2) {
                const uint64_t outs = (uint64_t)part_max_out(parts);
                const uint64_t frames = hs.mode == RS_PASSTHROUGH ? outs : (outs * hs.p + hs.q - 1) / hs.q;
                if (hs.desc.channels <= 2 && (frames + 8) * hs.desc.channels * bps + 32 <= (uint64_t)STAGE_BYTES) d.staged = (uint32_t)parts;
            }
        }
        if (d.staged == 4u) sb.quarters = true;
        if (!(hs.desc.channels == 1 && hs.desc.format == AF_FMT_F32 && hs.mode != RS_PASSTHROUGH && hs.p == 3 && hs.q == 1)) sb.split = true;
        // positions repeat every q outputs (p inputs): the first table-mode rate of the batch gets the kernel's position table
        if (hs.mode == RS_TABLE && sb.per_q == 0 && hs.q <= (uint32_t)KOFF_MAX && hs.q % 4 == 0 && STEP_SAMPLES % hs.q == 0 && hs.p < 65536) {
            sb.per_p = hs.p; sb.per_q = hs.q;
        }
        d.tile_begin = (uint32_t)sb.h_tiles.size();
        d.n_tiles = (hs.n_out + TILE_SAMPLES - 1) / TILE_SAMPLES;
        for (uint32_t t = 0; t < d.n_tiles; ++t) {
            TileDev td;
            plan_tile(d, (uint32_t)i, t, &td);                  // positions and stage fills: no 64-bit divisions in the kernel
            sb.h_tiles.push_back(td);
        }
        nf[i] = hs.n_frames; nv[i] = hs.n_vad_frames;
    }
    {   // a stream's last tile is often short: lay the tiles out so that every CTA of the launch (run_sub) gets a near-equal
        // share of the steps -- the kernel ends with its busiest CTA
        std::vector<uint32_t> steps(sb.h_tiles.size());
        for (size_t t = 0; t < steps.size(); ++t) steps[t] = sb.h_tiles[t].n_steps;
        const std::vector<uint32_t> order = balance_tile_order(steps, (uint32_t)std::min<size_t>(steps.size(), (size_t)cur_ctx().sm_count));
        std::vector<TileDev> planned;
        planned.swap(sb.h_tiles);
        sb.h_tiles.reserve(planned.size());
        for (const uint32_t t : order) sb.h_tiles.push_back(planned[t]);
    }
    AF_CUDA(sb.d_streams.grow(sb.count));
    AF_CUDA(sb.d_tiles.grow(sb.h_tiles.size() + 1));
    AF_CUDA(sb.d_nframes.grow(sb.count));
    AF_CUDA(sb.d_nvad.grow(sb.count));
    AF_CUDA(cudaMemcpy(sb.d_streams.get(), sb.h_streams.data(), sb.count * sizeof(StreamDev), cudaMemcpyHostToDevice));
    if (!sb.h_tiles.empty())
        AF_CUDA(cudaMemcpy(sb.d_tiles.get(), sb.h_tiles.data(), sb.h_tiles.size() * sizeof(TileDev), cudaMemcpyHostToDevice));
    AF_CUDA(cudaMemcpy(sb.d_nframes.get(), nf.data(), sb.count * sizeof(uint32_t), cudaMemcpyHostToDevice));
    AF_CUDA(cudaMemcpy(sb.d_nvad.get(), nv.data(), sb.count * sizeof(uint32_t), cudaMemcpyHostToDevice));
    return AF_OK;
}

// enqueue the kernels of sub-batch g on `st`; all pointers are device pointers of rows [0, sb.count)
int run_sub(af_batch *b, size_t g, float *pcm, uint64_t pcm_stride, float *logmel, uint64_t logmel_stride,
            uint8_t *vad, uint64_t vad_stride, float *energy, uint64_t energy_stride, VadState *vad_final,
            cudaStream_t st)
{
    const af_pipeline_config &cfg = b->pipe->cfg;
    const bool stft_vad = cfg.vad_enable && cfg.vad_frame_len == 0;
    const bool custom_vad = cfg.vad_enable && cfg.vad_frame_len != 0;
    SubBatch &sb = b->subs[g];
    const SubBatch &fp = b->poly ? b->poly->subs[g] : sb;     // what the fused kernel reads: the FIR's rows or the input
    if (b->poly && b->poly->jobs[g].n_tiles) {
        AF_CUDA(launch_polyphase_fir(b->poly->jobs[g], st));
        count_launch();
    }
    if (!fp.h_tiles.empty()) {
        FusedParams P{};
        P.streams = fp.d_streams.get(); P.tiles = fp.d_tiles.get(); P.n_tiles = (uint32_t)fp.h_tiles.size();
        P.fft = cur_ctx().d_fft.get(); P.mel = b->d_mel;
        P.pcm = pcm; P.pcm_stride = pcm_stride;
        P.logmel = cfg.n_mels ? logmel : nullptr; P.logmel_stride = logmel_stride;
        P.energy = stft_vad ? energy : nullptr; P.energy_stride = energy_stride;
        P.n_mels = (cfg.n_mels && logmel) ? cfg.n_mels : 0;
        P.do_energy = stft_vad ? 1 : 0;
        P.log_floor = cfg.log_floor;
        P.log_scale = cfg.log10 ? 0.30102999566398120f : 0.69314718055994531f;   // log10(2) : ln(2)
        P.use_stage = kernel_variant() == "sync" ? 0u : 1u;
        P.layout = fused_layout(stft_vad);
        P.quarters = fp.quarters ? 1u : 0u;
        P.neg_zero = -0.0f;
        P.per_p = fp.per_p; P.per_q = fp.per_q;
        const int n_ctas = (int)std::min<size_t>(fp.h_tiles.size(), (size_t)cur_ctx().sm_count);   // one persistent CTA per SM
        AF_CUDA(launch_fused(P, n_ctas, st, fp.split));
        count_launch();
    }
    if (custom_vad) {
        EnergyJob ej{};
        ej.y = pcm; ej.y_stride = pcm_stride; ej.n_frames = sb.d_nvad.get(); ej.n_frames_all = (uint32_t)b->max_vad;
        ej.frame_len = cfg.vad_frame_len; ej.hop = cfg.vad_hop; ej.energy = energy; ej.energy_stride = energy_stride;
        ej.n_streams = (uint32_t)sb.count;
        AF_CUDA(launch_frame_energy(ej, st));
        count_launch();
    }
    if (cfg.vad_enable) {
        ScanJob sj{};
        sj.energy = energy; sj.energy_stride = energy_stride; sj.n_frames = sb.d_nvad.get(); sj.n_frames_all = 0;
        sj.states = vad; sj.states_stride = vad_stride; sj.state_io = nullptr; sj.final_out = vad_final;
        sj.prm = b->pipe->vad_prm; sj.n_streams = (uint32_t)sb.count;
        sj.recs = sb.d_recs.get(); sj.n_seq = sb.n_seq;
        if (b->max_vad > 16384 && b->max_vad < 0x40000000ull) {              // long streams: many CTAs per stream
            AF_CUDA(sb.d_scan.grow(sb.count * scan_scratch_words((uint32_t)b->max_vad)));
            sj.max_frames = (uint32_t)b->max_vad; sj.scratch = sb.d_scan.get();
        }
        AF_CUDA(launch_vad_scan(sj, st));
        count_launch(scan_launches(sj));
    }
    return AF_OK;
}

uint64_t round_up(uint64_t v, uint64_t m) { return (v + m - 1) / m * m; }

// n elements of T, but no fewer than 256 bytes
template <class T> size_t min256(size_t n) { return std::max<size_t>(n, (256 + sizeof(T) - 1) / sizeof(T)); }

}  // namespace

extern "C" {

AF_API void af_pipeline_config_default(af_pipeline_config *cfg)
{
    if (!cfg) return;
    memset(cfg, 0, sizeof(*cfg));
    cfg->n_mels = 80;
    cfg->f_min = 0.0f; cfg->f_max = 8000.0f;
    cfg->log_floor = 1e-10f;
    cfg->log10 = 0;
    cfg->vad_enable = 1;
    af_vad_config_default(&cfg->vad);
    cfg->vad_frame_len = 0; cfg->vad_hop = 0;
    cfg->write_pcm = 1;
    cfg->pcm16 = 0;
}

AF_API int af_pipeline_create(const af_pipeline_config *cfg, af_pipeline **out)
{
    if (!out) return fail(AF_ERR_INVALID, "null out pointer");
    int rc = require_ctx();
    if (rc) return rc;
    af_pipeline_config c;
    if (cfg) c = *cfg; else af_pipeline_config_default(&c);
    if (c.n_mels > MAX_MELS) return fail(AF_ERR_INVALID, "n_mels %u > %d", c.n_mels, MAX_MELS);
    if (c.vad_enable && c.vad_frame_len != 0 && c.vad_hop == 0) return fail(AF_ERR_INVALID, "vad_hop must be positive");
    if (c.n_mels && !(c.f_max > c.f_min && c.f_min >= 0.0f)) return fail(AF_ERR_INVALID, "bad mel band [%g, %g]", c.f_min, c.f_max);
    af_pipeline *p = new af_pipeline;
    p->cfg = c;
    p->vad_prm = make_vad_params(c.vad);
    if (c.n_mels) {
        if (!build_mel_tables(c.n_mels, c.f_min, c.f_max, &p->h_mel)) { delete p; return fail(AF_ERR_INVALID, "mel table construction failed"); }
        if (!pipe_mel(p)) { delete p; return AF_ERR_CUDA; }
    }
    *out = p;
    return AF_OK;
}

AF_API void af_pipeline_destroy(af_pipeline *p)
{
    if (!p) return;
    for (int d = 0; d < MAX_DEV; ++d)
        if (p->d_mel[d].get() && device_ctx(d)) { DevScope scope_(d); p->d_mel[d].reset(); }
    delete p;
}

AF_API void af_batch_destroy(af_batch *b)
{
    if (!b) return;
    DevScope scope_(b->device);
    cudaDeviceSynchronize();
    for (auto &s : b->slots)
        if (s.st) cudaStreamDestroy(s.st);
    delete b;
}

AF_API int af_batch_create(af_pipeline *p, const af_stream_desc *streams, size_t n_streams, int mem, af_batch **out)
{
    if (!p || !out || (!streams && n_streams)) return fail(AF_ERR_INVALID, "null argument");
    if (mem != AF_MEM_DEVICE && mem != AF_MEM_HOST) return fail(AF_ERR_INVALID, "bad memory kind %d", mem);
    int rc = require_ctx();
    if (rc) return rc;
    // device batches run on the GPU that holds their input (every stream must live on the same one); host batches on
    // the calling thread's device
    int device = cur_device();
    if (mem == AF_MEM_DEVICE) {
        int owner = -1;
        for (size_t i = 0; i < n_streams; ++i) {
            if (!streams[i].data) continue;
            const int d = device_of_pointer(streams[i].data);
            if (d < 0) continue;
            if (owner < 0) owner = d;
            else if (owner != d) return fail(AF_ERR_INVALID, "stream %zu lives on GPU %d, stream(s) before it on GPU %d: one batch, one GPU (see af_sharded_batch_create)", i, d, owner);
        }
        if (owner >= 0) {
            rc = init_device(owner);
            if (rc) return rc;
            device = owner;
        }
    }
    AF_SCOPE(device);
    // (af_batch_destroy frees the slots, tables and streams allocated so far on every early return)
    std::unique_ptr<af_batch, void (*)(af_batch *)> b(new af_batch, af_batch_destroy);
    b->pipe = p; b->mem = mem; b->device = device;
    if (p->cfg.n_mels && !(b->d_mel = pipe_mel(p))) return AF_ERR_CUDA;
    b->streams.resize(n_streams);
    const af_pipeline_config &cfg = p->cfg;
    for (size_t i = 0; i < n_streams; ++i) {
        HostStream &hs = b->streams[i];
        hs.desc = streams[i];
        const af_stream_desc &d = hs.desc;
        if (d.channels == 0) return fail(AF_ERR_INVALID, "stream %zu: channels must be >= 1", i);
        if (d.format != AF_FMT_F32 && d.format != AF_FMT_I16) return fail(AF_ERR_INVALID, "stream %zu: bad format %u", i, d.format);
        if (!d.data && d.n_samples) return fail(AF_ERR_INVALID, "stream %zu: null data", i);
        if (mem == AF_MEM_DEVICE && ((uintptr_t)d.data & 15)) return fail(AF_ERR_INVALID, "stream %zu: device data must be 16-byte aligned", i);
        const uint64_t n_in = (d.n_samples + d.channels - 1) / d.channels;
        if (n_in >= (1ull << 31)) return fail(AF_ERR_INVALID, "stream %zu: too long (%llu frames)", i, (unsigned long long)n_in);
        uint64_t n_out = 0;
        rc = plan_rate(d.sample_rate, OUT_RATE, n_in, &n_out, &hs.mode, &hs.p, &hs.q, &hs.table);
        if (rc) return rc;
        if (n_out >= (1ull << 31)) return fail(AF_ERR_INVALID, "stream %zu: output too long", i);
        if (hs.mode != RS_PASSTHROUGH &&
            (uint64_t)(TILE_SAMPLES + YLEN + FUSED_THREADS) * hs.p + hs.q >= (1ull << 32))
            return fail(AF_ERR_RESAMPLING_FAILED, "stream %zu: unsupported rate ratio %u/%u", i, hs.p, hs.q);
        hs.n_in = (uint32_t)n_in; hs.n_out = (uint32_t)n_out;
        hs.n_frames = n_out >= WIN ? (uint32_t)(1 + (n_out - WIN) / HOP) : 0;
        if (!cfg.vad_enable) hs.n_vad_frames = 0;
        else if (cfg.vad_frame_len == 0) hs.n_vad_frames = hs.n_frames;
        else hs.n_vad_frames = n_out >= cfg.vad_frame_len ? (uint32_t)(1 + (n_out - cfg.vad_frame_len) / cfg.vad_hop) : 0;
        b->max_out = std::max<uint64_t>(b->max_out, hs.n_out);
        b->max_frames = std::max<uint64_t>(b->max_frames, hs.n_frames);
        b->max_vad = std::max<uint64_t>(b->max_vad, hs.n_vad_frames);
    }
    b->pcm_stride = round_up(std::max<uint64_t>(b->max_out, 4), 4);
    b->logmel_stride = round_up(std::max<uint64_t>(b->max_frames * cfg.n_mels, 4), 4);
    b->vad_stride = round_up(std::max<uint64_t>(b->max_vad, 16), 16);
    b->energy_stride = round_up(std::max<uint64_t>(b->max_vad, 4), 4);

    if (mem == AF_MEM_DEVICE) {
        b->subs.resize(1);
        b->subs[0].first = 0; b->subs[0].count = n_streams;
        if (n_streams) { rc = build_sub(b->streams, b->subs[0], nullptr); if (rc) return rc; }
    } else {
        // host mode: groups of streams of ~32 MB input (measured: 96 MB 29.4 ms, 32 MB 28.3 ms per cfg2 batch against a
        // PCIe ceiling of 28.1 ms on the box), cycled through 3 slots so that the H2D copy of
        // group g+1, the kernels of group g and the D2H copy of group g-1 overlap
        // (AF_HOST_SUB_MB / AF_HOST_SLOTS override the defaults: experiments)
        static const size_t sub_mb = [] { const char *e = getenv("AF_HOST_SUB_MB"); return e ? (size_t)atoi(e) : (size_t)32; }();
        static const size_t want_slots = [] { const char *e = getenv("AF_HOST_SLOTS"); return e ? (size_t)atoi(e) : (size_t)3; }();
        const size_t target = std::max<size_t>(sub_mb, 1) << 20;
        size_t i = 0;
        while (i < n_streams) {
            SubBatch sb;
            sb.first = i;
            size_t bytes = 0;
            while (i < n_streams && (sb.count == 0 || bytes < target)) {
                const af_stream_desc &d = b->streams[i].desc;
                const size_t sz = d.n_samples * (d.format == AF_FMT_I16 ? 2 : 4);
                sb.in_off.push_back(bytes);
                bytes += round_up(sz, 256);
                sb.count++; i++;
            }
            sb.in_bytes = bytes;
            b->subs.push_back(std::move(sb));
        }
        size_t max_rows = 0, max_in = 0;
        for (auto &sb : b->subs) { max_rows = std::max(max_rows, sb.count); max_in = std::max(max_in, sb.in_bytes); }
        b->slot_rows = max_rows;
        const size_t n_slots = std::min<size_t>(std::max<size_t>(want_slots, 1), std::max<size_t>(1, b->subs.size()));
        b->slots.resize(n_slots);
        for (auto &s : b->slots) {
            AF_CUDA(cudaStreamCreateWithFlags(&s.st, cudaStreamNonBlocking));
            AF_CUDA(s.d_in.alloc(min256<char>(max_in)));
            AF_CUDA(s.d_pcm.alloc(min256<float>(max_rows * b->pcm_stride)));
            if (cfg.pcm16) AF_CUDA(s.d_pcm16.alloc(min256<int16_t>(max_rows * b->pcm_stride)));
            if (cfg.n_mels) AF_CUDA(s.d_logmel.alloc(min256<float>(max_rows * b->logmel_stride)));
            if (cfg.vad_enable) {
                AF_CUDA(s.d_vad.alloc(min256<uint8_t>(max_rows * b->vad_stride)));
                AF_CUDA(s.d_energy.alloc(min256<float>(max_rows * b->energy_stride)));
                AF_CUDA(s.d_final.alloc(min256<VadState>(max_rows)));
            }
        }
        for (size_t g = 0; g < b->subs.size(); ++g) {
            rc = build_sub(b->streams, b->subs[g], b->slots[g % n_slots].d_in.get());
            if (rc) return rc;
        }
    }
    *out = b.release();
    return AF_OK;
}

AF_API size_t af_batch_n_streams(const af_batch *b) { return b ? b->streams.size() : 0; }

AF_API int af_batch_counts(const af_batch *b, uint32_t *n_out, uint32_t *n_feat_frames, uint32_t *n_vad_frames)
{
    if (!b) return fail(AF_ERR_INVALID, "null batch");
    for (size_t i = 0; i < b->streams.size(); ++i) {
        if (n_out) n_out[i] = b->streams[i].n_out;
        if (n_feat_frames) n_feat_frames[i] = b->pipe->cfg.n_mels ? b->streams[i].n_frames : 0;
        if (n_vad_frames) n_vad_frames[i] = b->streams[i].n_vad_frames;
    }
    return AF_OK;
}

AF_API int af_batch_strides(const af_batch *b, uint64_t *pcm_stride, uint64_t *logmel_stride, uint64_t *vad_stride)
{
    if (!b) return fail(AF_ERR_INVALID, "null batch");
    if (pcm_stride) *pcm_stride = b->pcm_stride;
    if (logmel_stride) *logmel_stride = b->logmel_stride;
    if (vad_stride) *vad_stride = b->vad_stride;
    return AF_OK;
}

static int check_outputs(const af_batch *b, const af_outputs *o)
{
    const af_pipeline_config &cfg = b->pipe->cfg;
    if (!o) return fail(AF_ERR_INVALID, "null outputs");
    // the fused kernel stores PCM and log-mel rows with 16-byte vector stores
    if (o->pcm && b->mem == AF_MEM_DEVICE && (reinterpret_cast<uintptr_t>(o->pcm) & 15)) return fail(AF_ERR_INVALID, "device pcm pointer must be 16-byte aligned");
    if (o->pcm && (o->pcm_stride < b->max_out || (o->pcm_stride & 3))) return fail(AF_ERR_CAPACITY, "pcm_stride %llu too small or not a multiple of 4 (need >= %llu)", (unsigned long long)o->pcm_stride, (unsigned long long)b->max_out);
    if (o->logmel && cfg.n_mels && (o->logmel_stride < b->max_frames * cfg.n_mels || (o->logmel_stride & 3))) return fail(AF_ERR_CAPACITY, "logmel_stride too small or not a multiple of 4");
    if (o->vad && o->vad_stride < b->max_vad) return fail(AF_ERR_CAPACITY, "vad_stride too small");
    if (o->energy && o->energy_stride < b->max_vad) return fail(AF_ERR_CAPACITY, "energy_stride too small");
    return AF_OK;
}

}  // extern "C"

namespace afrt {

int batch_device(const af_batch *b) { return b ? b->device : -1; }
int batch_check_outputs(const af_batch *b, const af_outputs *o) { return check_outputs(b, o); }
const af_pipeline_config &pipeline_cfg(const af_pipeline *p) { return p->cfg; }

// the counts af_batch_create derives for one stream, without creating anything on a device (a rank plans the streams of
// the other ranks this way: every rank knows every row of the gathered result)
int plan_stream_counts(const af_pipeline_config &cfg, const af_stream_desc &d, uint32_t *n_out_, uint32_t *n_frames_, uint32_t *n_vad_)
{
    if (d.channels == 0) return fail(AF_ERR_INVALID, "channels must be >= 1");
    const uint64_t n_in = (d.n_samples + d.channels - 1) / d.channels;
    if (n_in >= (1ull << 31)) return fail(AF_ERR_INVALID, "stream too long (%llu frames)", (unsigned long long)n_in);
    uint64_t n_out = 0; uint32_t mode, p, q;
    int rc = plan_rate(d.sample_rate, OUT_RATE, n_in, &n_out, &mode, &p, &q, nullptr);
    if (rc) return rc;
    if (n_out >= (1ull << 31)) return fail(AF_ERR_INVALID, "output too long");
    const uint32_t n_frames = n_out >= WIN ? (uint32_t)(1 + (n_out - WIN) / HOP) : 0;
    uint32_t n_vad = 0;
    if (!cfg.vad_enable) n_vad = 0;
    else if (cfg.vad_frame_len == 0) n_vad = n_frames;
    else n_vad = n_out >= cfg.vad_frame_len ? (uint32_t)(1 + (n_out - cfg.vad_frame_len) / cfg.vad_hop) : 0;
    if (n_out_) *n_out_ = (uint32_t)n_out;
    if (n_frames_) *n_frames_ = n_frames;
    if (n_vad_) *n_vad_ = n_vad;
    return AF_OK;
}
uint64_t batch_max_vad(const af_batch *b) { return b ? b->max_vad : 0; }

// the body of af_batch_run: enqueues on `st` (the batch's device must be current), never synchronises; the VAD states
// go to `vad` / `vad_stride`, which the sharded batches point into their gather buffer
int batch_run_on(af_batch *b, const af_outputs *o, uint8_t *vad, uint64_t vad_stride, cudaStream_t st)
{
    if (b->streams.empty()) return AF_OK;
    const af_pipeline_config &cfg = b->pipe->cfg;
    const size_t S = b->streams.size();
    float *energy = o->energy; uint64_t energy_stride = o->energy_stride;
    if (cfg.vad_enable && !energy) {
        AF_CUDA(b->d_energy.grow(min256<float>(S * b->energy_stride)));
        energy = b->d_energy.get(); energy_stride = b->energy_stride;
    }
    float *pcm = cfg.write_pcm ? o->pcm : nullptr; uint64_t pcm_stride = o->pcm_stride;
    const bool wire16 = cfg.pcm16 && pcm;                        // PCM leaves as i16 wire samples: f32 rows stay internal
    if (wire16) pcm = nullptr;
    if ((wire16 || (cfg.vad_enable && cfg.vad_frame_len != 0)) && !pcm) {      // custom VAD frames read the PCM back
        AF_CUDA(b->d_pcm_scratch.grow(min256<float>(S * b->pcm_stride)));
        pcm = b->d_pcm_scratch.get(); pcm_stride = b->pcm_stride;
    }
    int rc = run_sub(b, 0, pcm, pcm_stride, o->logmel, o->logmel_stride, vad, vad_stride, energy, energy_stride,
                     reinterpret_cast<VadState *>(o->vad_final), st);
    if (rc) return rc;
    if (wire16) {                                                // websocket.rs:246-251 on the rows, 2 bytes per sample out
        AF_CUDA(launch_pcm16_rows(pcm, pcm_stride, reinterpret_cast<int16_t *>(o->pcm), o->pcm_stride, (uint32_t)b->max_out, (uint32_t)S, st));
        count_launch();
    }
    return AF_OK;
}

}  // namespace afrt

extern "C" {

AF_API int af_batch_run(af_batch *b, const af_outputs *o, void *cuda_stream)
{
    if (!b) return fail(AF_ERR_INVALID, "null batch");
    if (b->mem != AF_MEM_DEVICE) return fail(AF_ERR_INVALID, "batch was planned for host buffers; use af_batch_run_host");
    int rc = check_outputs(b, o);
    if (rc) return rc;
    AF_SCOPE(b->device);
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : cur_ctx().stream;
    rc = batch_run_on(b, o, o->vad, o->vad_stride, st);
    if (rc) return rc;
    if (!cuda_stream) AF_CUDA(cudaStreamSynchronize(st));
    return AF_OK;
}

AF_API int af_batch_run_host(af_batch *b, const af_outputs *o)
{
    if (!b) return fail(AF_ERR_INVALID, "null batch");
    if (b->mem != AF_MEM_HOST) return fail(AF_ERR_INVALID, "batch was planned for device buffers; use af_batch_run");
    int rc = check_outputs(b, o);
    if (rc) return rc;
    AF_SCOPE(b->device);
    const af_pipeline_config &cfg = b->pipe->cfg;
    const size_t n_slots = b->slots.size();
    for (size_t g = 0; g < b->subs.size(); ++g) {
        SubBatch &sb = b->subs[g];
        af_batch::Slot &sl = b->slots[g % n_slots];
        cudaStream_t st = sl.st;
        // host -> device: one copy per run of streams that are contiguous on both sides (rows of one host array are)
        for (size_t i = 0; i < sb.count;) {
            const af_stream_desc &d0 = b->streams[sb.first + i].desc;
            size_t bytes = d0.n_samples * (d0.format == AF_FMT_I16 ? 2 : 4);
            const size_t bytes0 = bytes;
            size_t j = i + 1;
            while (!sb.no_merge && j < sb.count) {
                const af_stream_desc &dj = b->streams[sb.first + j].desc;
                if ((const char *)dj.data != (const char *)d0.data + bytes || sb.in_off[j] != sb.in_off[i] + bytes) break;
                bytes += dj.n_samples * (dj.format == AF_FMT_I16 ? 2 : 4);
                ++j;
            }
            if (bytes) {
                cudaError_t ce = cudaMemcpyAsync(sl.d_in.get() + sb.in_off[i], d0.data, bytes, cudaMemcpyHostToDevice, st);
                if (ce == cudaErrorInvalidValue && j > i + 1) {
                    // rows that happen to be adjacent in host memory but belong to separate pinned allocations: CUDA refuses a
                    // copy that spans two of them.  Not sticky: copy this sub-batch stream by stream from now on.
                    (void)cudaGetLastError();
                    sb.no_merge = true;
                    j = i + 1;
                    ce = bytes0 ? cudaMemcpyAsync(sl.d_in.get() + sb.in_off[i], d0.data, bytes0, cudaMemcpyHostToDevice, st) : cudaSuccess;
                }
                AF_CUDA(ce);
            }
            i = j;
        }
        const bool need_pcm = (cfg.write_pcm && o->pcm) || (cfg.vad_enable && cfg.vad_frame_len != 0);
        rc = run_sub(b, g, need_pcm ? sl.d_pcm.get() : nullptr, b->pcm_stride, sl.d_logmel.get(), b->logmel_stride, sl.d_vad.get(),
                     b->vad_stride, sl.d_energy.get(), b->energy_stride, sl.d_final.get(), st);
        if (rc) return rc;
        const size_t r0 = sb.first;
        if (cfg.write_pcm && o->pcm && cfg.pcm16) {
            AF_CUDA(launch_pcm16_rows(sl.d_pcm.get(), b->pcm_stride, sl.d_pcm16.get(), b->pcm_stride, (uint32_t)b->max_out, (uint32_t)sb.count, st));
            count_launch();
            int16_t *dst = reinterpret_cast<int16_t *>(o->pcm);
            AF_CUDA(cudaMemcpy2DAsync(dst + r0 * o->pcm_stride, o->pcm_stride * sizeof(int16_t), sl.d_pcm16.get(),
                                      b->pcm_stride * sizeof(int16_t), b->max_out * sizeof(int16_t), sb.count,
                                      cudaMemcpyDeviceToHost, st));
        } else if (cfg.write_pcm && o->pcm)
            AF_CUDA(cudaMemcpy2DAsync(o->pcm + r0 * o->pcm_stride, o->pcm_stride * sizeof(float), sl.d_pcm.get(),
                                      b->pcm_stride * sizeof(float), b->max_out * sizeof(float), sb.count,
                                      cudaMemcpyDeviceToHost, st));
        if (cfg.n_mels && o->logmel && b->max_frames)
            AF_CUDA(cudaMemcpy2DAsync(o->logmel + r0 * o->logmel_stride, o->logmel_stride * sizeof(float), sl.d_logmel.get(),
                                      b->logmel_stride * sizeof(float), b->max_frames * cfg.n_mels * sizeof(float),
                                      sb.count, cudaMemcpyDeviceToHost, st));
        if (cfg.vad_enable && b->max_vad) {
            if (o->vad)
                AF_CUDA(cudaMemcpy2DAsync(o->vad + r0 * o->vad_stride, o->vad_stride, sl.d_vad.get(), b->vad_stride, b->max_vad,
                                          sb.count, cudaMemcpyDeviceToHost, st));
            if (o->energy)
                AF_CUDA(cudaMemcpy2DAsync(o->energy + r0 * o->energy_stride, o->energy_stride * sizeof(float), sl.d_energy.get(),
                                          b->energy_stride * sizeof(float), b->max_vad * sizeof(float), sb.count,
                                          cudaMemcpyDeviceToHost, st));
        }
        if (cfg.vad_enable && o->vad_final)
            AF_CUDA(cudaMemcpyAsync(o->vad_final + r0, sl.d_final.get(), sb.count * sizeof(VadState), cudaMemcpyDeviceToHost, st));
    }
    for (auto &sl : b->slots) AF_CUDA(cudaStreamSynchronize(sl.st));
    return AF_OK;
}

AF_API int af_batch_set_vad_configs(af_batch *b, const af_vad_config *cfgs)
{
    if (!b) return fail(AF_ERR_INVALID, "null batch");
    if (!b->pipe->cfg.vad_enable) return fail(AF_ERR_INVALID, "the pipeline runs no VAD (vad_enable == 0)");
    AF_SCOPE(b->device);
    const size_t S = b->streams.size();
    const ScanRec base = scan_rec(b->pipe->vad_prm);
    std::vector<ScanRec> recs;
    bool custom = false;                          // some stream differs from the pipeline: the scan takes the records
    if (cfgs && S) {
        recs.resize(S);
        make_scan_recs(cfgs, S, recs.data());
        for (size_t k = 0; k < S && !custom; ++k) custom = !same_rec(recs[k], base);
    }
    // every sub-batch's slice is allocated before anything changes
    std::vector<DevBuf<ScanRec>> d(b->subs.size());
    std::vector<uint32_t> n_seq(b->subs.size(), 0);
    if (custom)
        for (size_t g = 0; g < b->subs.size(); ++g) {
            const SubBatch &sb = b->subs[g];
            AF_CUDA(d[g].alloc(sb.count));
            for (size_t i = 0; i < sb.count; ++i) n_seq[g] += recs[sb.first + i].seq;
        }
    AF_CUDA(cudaDeviceSynchronize());             // runs still in flight on the caller's streams read the old slices
    if (custom)
        for (size_t g = 0; g < b->subs.size(); ++g)
            AF_CUDA(cudaMemcpy(d[g].get(), recs.data() + b->subs[g].first, b->subs[g].count * sizeof(ScanRec),
                               cudaMemcpyHostToDevice));
    for (size_t g = 0; g < b->subs.size(); ++g) {
        b->subs[g].d_recs = std::move(d[g]);
        b->subs[g].n_seq = n_seq[g];
    }
    return AF_OK;
}

AF_API int af_batch_set_resampler(af_batch *b, uint32_t filter)
{
    if (!b) return fail(AF_ERR_INVALID, "null batch");
    if (filter != AF_RESAMPLE_CUBIC && filter != AF_RESAMPLE_POLYPHASE) return fail(AF_ERR_INVALID, "unknown resampling filter %u", filter);
    const size_t S = b->streams.size();
    for (size_t i = 0; i < S && filter == AF_RESAMPLE_POLYPHASE; ++i) {
        uint32_t p, q;
        if (!polyphase_ratio(b->streams[i].desc.sample_rate, OUT_RATE, &p, &q))
            return fail(AF_ERR_RESAMPLING_FAILED, "stream %zu: %u Hz -> %d Hz reduces to %u / %u; the polyphase filter takes max(p, q) <= %d",
                        i, b->streams[i].desc.sample_rate, OUT_RATE, p, q, POLY_MAX_RATIO);
    }
    AF_SCOPE(b->device);
    if (filter == AF_RESAMPLE_CUBIC) {
        if (b->poly) {
            AF_CUDA(cudaDeviceSynchronize());     // runs still in flight read the rows
            b->poly.reset();
        }
        return AF_OK;
    }
    // everything is built before anything changes
    auto ph = std::make_unique<Polyphase>();
    std::map<uint32_t, std::vector<float>> h_taps;
    for (const HostStream &hs : b->streams) {
        const uint32_t rate = hs.desc.sample_rate;
        if (h_taps.count(rate)) continue;
        uint32_t p, q;
        polyphase_ratio(rate, OUT_RATE, &p, &q);
        polyphase_filter(p, q, &h_taps[rate]);
        const std::vector<float> &h = h_taps[rate];
        AF_CUDA(ph->taps[rate].alloc(h.size()));
        AF_CUDA(cudaMemcpy(ph->taps[rate].get(), h.data(), h.size() * sizeof(float), cudaMemcpyHostToDevice));
    }
    ph->rows.resize(S);
    for (size_t i = 0; i < S; ++i) {
        const HostStream &hs = b->streams[i];
        HostStream &r = ph->rows[i];
        r = hs;
        r.desc.data = nullptr; r.desc.n_samples = hs.n_out; r.desc.sample_rate = OUT_RATE;
        r.desc.channels = 1; r.desc.format = AF_FMT_F32;
        r.n_in = hs.n_out; r.mode = RS_PASSTHROUGH; r.p = r.q = 1; r.table.reset();
    }
    const size_t n_blocks = b->mem == AF_MEM_DEVICE ? 1 : b->slots.size();
    const size_t block_rows = b->mem == AF_MEM_DEVICE ? S : b->slot_rows;
    ph->d_rows.resize(n_blocks);
    for (auto &d : ph->d_rows) AF_CUDA(d.alloc(min256<float>(block_rows * b->pcm_stride)));
    const size_t G = b->subs.size();
    ph->subs.resize(G); ph->jobs.resize(G); ph->d_fir.resize(G); ph->d_tiles.resize(G);
    for (size_t g = 0; g < G; ++g) {
        const SubBatch &sb = b->subs[g];
        float *rows = ph->d_rows[g % n_blocks].get();
        const char *in_base = b->mem == AF_MEM_DEVICE ? nullptr : b->slots[g % b->slots.size()].d_in.get();
        SubBatch &fp = ph->subs[g];
        fp.first = sb.first; fp.count = sb.count;
        std::vector<FirStream> fs(sb.count);
        std::vector<uint2> tiles;
        FirJob &J = ph->jobs[g];
        J = FirJob{};
        for (size_t i = 0; i < sb.count; ++i) {
            const HostStream &hs = b->streams[sb.first + i];
            FirStream &f = fs[i];
            memset(&f, 0, sizeof(f));
            f.data = in_base ? (const void *)(in_base + sb.in_off[i]) : hs.desc.data;
            f.n_samples = hs.desc.n_samples; f.n_in = hs.n_in; f.n_out = hs.n_out;
            f.channels = hs.desc.channels; f.format = hs.desc.format;
            polyphase_ratio(hs.desc.sample_rate, OUT_RATE, &f.p, &f.q);
            f.L = 10 * std::max(f.p, f.q);
            f.tile_out = fir_tile_outputs(f.p, f.q);
            f.h = ph->taps[hs.desc.sample_rate].get();
            f.y = rows + i * b->pcm_stride;
            f.taps_smem = 2 * f.L + 1 <= (uint32_t)FIR_TAPS_SMEM ? 1u : 0u;
            if (f.p == 3 && f.q == 1) memcpy(J.h3, h_taps[hs.desc.sample_rate].data(), sizeof(J.h3));
            const uint32_t n_tiles = (hs.n_out + f.tile_out - 1) / f.tile_out;
            for (uint32_t t = 0; t < n_tiles; ++t) tiles.push_back(make_uint2((uint32_t)i, t));
            if (n_tiles) J.smem_floats = std::max<uint32_t>(J.smem_floats, (uint32_t)fir_smem_floats(f.p, f.q, f.taps_smem));
            fp.in_off.push_back(i * b->pcm_stride * sizeof(float));
        }
        AF_CUDA(ph->d_fir[g].alloc(std::max<size_t>(sb.count, 1)));
        AF_CUDA(ph->d_tiles[g].alloc(std::max<size_t>(tiles.size(), 1)));
        if (sb.count) AF_CUDA(cudaMemcpy(ph->d_fir[g].get(), fs.data(), sb.count * sizeof(FirStream), cudaMemcpyHostToDevice));
        if (!tiles.empty()) AF_CUDA(cudaMemcpy(ph->d_tiles[g].get(), tiles.data(), tiles.size() * sizeof(uint2), cudaMemcpyHostToDevice));
        J.streams = ph->d_fir[g].get(); J.tiles = ph->d_tiles[g].get(); J.n_tiles = (uint32_t)tiles.size();
        if (sb.count) {
            int rc = build_sub(ph->rows, fp, rows);
            if (rc) return rc;
        }
    }
    AF_CUDA(cudaDeviceSynchronize());             // runs still in flight read the previous rows
    b->poly = std::move(ph);
    return AF_OK;
}

AF_API size_t af_debug_polyphase_filter(uint32_t input_rate, uint32_t output_rate, float *h, size_t cap, uint32_t *p, uint32_t *q)
{
    uint32_t p_ = 0, q_ = 0;
    const bool ok = polyphase_ratio(input_rate, output_rate, &p_, &q_);
    if (p) *p = p_;
    if (q) *q = q_;
    if (!ok) return 0;
    std::vector<float> t;
    polyphase_filter(p_, q_, &t);
    for (size_t i = 0; i < t.size() && i < cap && h; ++i) h[i] = t[i];
    return t.size();
}

AF_API int af_pipeline_run(af_pipeline *p, const af_stream_desc *streams, size_t n_streams, const af_outputs *out)
{
    af_batch *b = nullptr;
    int rc = af_batch_create(p, streams, n_streams, AF_MEM_HOST, &b);
    if (rc) return rc;
    rc = af_batch_run_host(b, out);
    af_batch_destroy(b);
    return rc;
}

AF_API float af_debug_vad_energy_threshold(float threshold_db) { return vad_energy_threshold(threshold_db); }

AF_API size_t af_debug_resample_plan(uint32_t input_rate, uint32_t output_rate, size_t n_chunks, float *frac, size_t cap,
                                     int *mode)
{
    RsRecurrence r;
    r.init(input_rate, output_rate);
    if (mode) *mode = (int)r.mode();
    if (r.passthrough || r.end_idx <= 0) return 0;
    std::vector<float> f;
    for (size_t c = 0; c < n_chunks; ++c) r.step(&f);
    for (size_t i = 0; i < f.size() && i < cap; ++i) frac[i] = f[i];
    return f.size();
}

AF_API uint64_t af_debug_tile_order(const uint32_t *steps, size_t n, uint32_t n_ctas, uint32_t *order)
{
    const std::vector<uint32_t> st(steps, steps + n);
    const std::vector<uint32_t> o = balance_tile_order(st, n_ctas);
    std::copy(o.begin(), o.end(), order);
    return tile_order_max_steps(st, o, n_ctas);
}

}  // extern "C"

// ------------------------------------------------------------------------------------------
// streaming sessions (BASELINE config 5): n_streams streams, state resident on the device
// ------------------------------------------------------------------------------------------
struct af_session {
    af_pipeline *pipe = nullptr;
    int device = -1;                  // the GPU that holds the session state
    MelTables *d_mel = nullptr;
    size_t S = 0;
    // the capture formats the session admits (af_session_create: one); a stream's state names its format.  The buffers
    // are sized for the largest bound over the formats: max_tick_frames, max_new_y (below) and max_ring_samples
    struct Format { uint32_t rate, channels, max_tick_frames; };
    std::vector<Format> fmts;
    DevBuf<SessionFormat> d_fmts;                              // their device table, read by af_session_tick_streams_kernel
    bool any_table = false;                                    // some format resamples through a fraction table (RS_TABLE)
    uint32_t format = 0, max_tick_frames = 0;
    uint64_t max_ring_samples = 0;
    // input history: last 16 frames + residual (< 128), ping-pong
    DevBuf<float> in_buf[2]; uint64_t in_stride = 0; int in_cur = 0;
    // 16 kHz carry (samples not yet covered by an emitted frame), ping-pong
    DevBuf<float> y_buf[2]; uint64_t y_stride = 0; int y_cur = 0;
    uint32_t frame_len = WIN, hop = HOP;   // framing of the features / VAD
    bool framing = false;
    // packed ticks (STFT frames): the rows of y_buf are a whole number of hops apart, so `pk_rows` consecutive streams
    // read as ONE virtual stream whose frame slot r * pk_slots + j is frame j of row r (the slots >= T straddle rows and
    // are ignored).  A tick of two frames per stream then fills the fused kernel's 32-frame steps instead of leaving
    // 30 of 32 slots empty, and the tiles are planned once (the virtual streams never change length).
    bool packed = false;
    uint32_t pk_slots = 0, pk_rows = 0, pk_n = 0;          // frame slots per row, rows per virtual stream, virtual streams
    DevBuf<StreamDev> d_ptab[2];
    DevBuf<TileDev> d_ptiles[2];
    DevBuf<VadState> d_vad;
    DevBuf<float> d_energy; uint64_t energy_stride = 0;
    DevBuf<float> d_frac;
    DevBuf<char> d_in_stage;                                  // host-mode staging of the tick input
    DevBuf<float> d_lm; DevBuf<uint8_t> d_states;             // host-mode staging of outputs
    uint64_t lm_stride = 0, st_stride = 0;
    std::vector<float> frac_host;
    PinnedBuf<float> ring_stage;                              // pinned rows for af_session_push_rings
    // level metering (af_session_enable_levels): peak of the last tick per stream + the detector states, on the host
    struct Levels {
        DevBuf<float> d_peak;
        PinnedBuf<float> h_peak;
        PinnedBuf<VadState> h_vad;
    };
    Levels lv;
    bool levels = false, levels_valid = false;
    // wire output (af_session_enable_wire): device rows written by the wire kernel, pinned host copies for AF_MEM_HOST
    struct Wire {
        af_wire_config cfg{};
        DevBuf<int16_t> d_pcm16; PinnedBuf<int16_t> h_pcm16; uint64_t pcm16_stride = 0;   // int16_t elements
        DevBuf<char> d_b64; PinnedBuf<char> h_b64; uint64_t b64_stride = 0;               // bytes
        uint64_t cap = 0;                                                                 // payload samples a row holds
        DevBuf<WireTick> d_ticks;
        PinnedBuf<af_wire_tick> h_ticks;
        // wire features (af_session_enable_wire_features): the kept frames' log-mel rows and their counts; no rows: off.
        // valid: a push has filled them since they were built
        struct Features {
            int mem = AF_MEM_HOST;
            DevBuf<float> d_rows; PinnedBuf<float> h_rows; uint64_t stride = 0;          // floats
            DevBuf<uint32_t> d_n; PinnedBuf<uint32_t> h_n;
            bool valid = false;
        };
        Features feat;
        // pre-roll (af_session_set_wire_preroll): P frames; per stream a ring of the PCM16 hops (and, with features, the
        // log-mel rows) of up to P frames after its last payload frame, its count of valid frames and its next slot.
        // frames == 0: off, nothing allocated
        struct Preroll {
            uint32_t frames = 0;
            DevBuf<int16_t> d_pcm; DevBuf<float> d_lm;
            DevBuf<uint32_t> d_n, d_pos;
        };
        Preroll pre;
        // segment table (af_session_enable_wire_segments): per stream the pieces of the gated payload and their count;
        // no rows: off.  valid: a push has filled them since they were built
        struct Segments {
            int mem = AF_MEM_HOST;
            DevBuf<WireSegment> d_rows; PinnedBuf<af_wire_segment> h_rows; uint64_t stride = 0;   // entries
            DevBuf<uint32_t> d_n; PinnedBuf<uint32_t> h_n;
            bool valid = false;
        };
        Segments seg;
    };
    Wire wr;
    uint64_t max_new_y = 0;                                   // bound of the 16 kHz samples one tick produces
    bool wire = false, wire_valid = false;
    DevBuf<uint8_t> d_wire_prev;                              // per stream: state of the latest completed frame
    // the bookkeeping of one stream's timeline.  While !diverged, `shared` is the position of every stream and a tick of
    // equal counts takes the lockstep tick kernel; while diverged, ss[k] is stream k's position (af_session_push_streams).
    // The ping-pong buffers (in_cur, y_cur) flip for all streams on every tick either way.
    struct StreamState {
        RsRecurrence rec;                                      // the stream's f64 chunk recurrence
        uint32_t in_len;                                       // frames held in its row of in_buf[in_cur]
        // frames / samples at the front of the current rows that the NEXT tick's ingest / resample skip: the compaction
        // after a tick costs no kernel of its own
        uint32_t in_drop, y_drop;
        uint32_t y_len;                                        // 16 kHz carry held in its row of y_buf[y_cur]
        long long in_base;                                     // global frame index of the row's first frame
        uint64_t frames_emitted;
        bool restart;                                          // start afresh at the next push (end / af_session_reset_streams)
        uint32_t fmt;                                          // index into fmts (of the next life while `restart`)
    };
    StreamState shared{};
    std::vector<StreamState> ss, ss_next;
    bool diverged = false;
    std::vector<uint32_t> plan_slots;                          // scratch: open-addressing table of the tick's distinct plans
    struct TickPlan {                                          // the tick's plan: [S] StreamTick, then [S] uint32 frame counts
        DevBuf<StreamTick> d;
        PinnedBuf<StreamTick> h;
    };
    TickPlan tick;
    DevBuf<float> d_pcm_stage;                                 // host-mode PCM rows of a per-stream tick
    std::vector<uint32_t> counts;                              // scratch: equal counts (af_session_push), ring reads
    std::vector<uint64_t> first_frames;                        // per stream: first frame completed by the last push
    // per-stream detector configurations (af_session_set_vad_configs), allocated by the first call: host records, their
    // device table, the range [recs_lo, recs_hi) set since the last upload, and how many records differ from the
    // pipeline's (0: the scan takes the pipeline's configuration, as a session that never set one)
    PinnedBuf<ScanRec> h_recs;
    DevBuf<ScanRec> d_recs;
    size_t recs_lo = 0, recs_hi = 0, n_custom_recs = 0;
    std::vector<af_vad_config> vad_cfgs;                       // the configurations h_recs was made from (a record carries one)
    // stream records (af_session_export_streams / af_session_import_streams), grown on demand: the per-stream move table,
    // the headers of device records, and the staging rows of host records' device parts
    struct Transfer {
        PinnedBuf<RecordMove> h_moves;
        DevBuf<RecordMove> d_moves;
        PinnedBuf<uint8_t> h_hdr;
        DevBuf<uint8_t> stage;
    };
    Transfer xfer;
};
static_assert(sizeof(WireTick) == sizeof(af_wire_tick) && offsetof(WireTick, started) == offsetof(af_wire_tick, started) &&
              offsetof(WireTick, in_speech) == offsetof(af_wire_tick, in_speech), "WireTick mirrors af_wire_tick");
static_assert(sizeof(af_wire_segment) == 16 && sizeof(WireSegment) == sizeof(af_wire_segment) &&
              offsetof(WireSegment, offset) == offsetof(af_wire_segment, offset) &&
              offsetof(WireSegment, n_frames) == offsetof(af_wire_segment, n_frames) &&
              offsetof(WireSegment, preroll) == offsetof(af_wire_segment, preroll) &&
              offsetof(WireSegment, flags) == offsetof(af_wire_segment, flags), "WireSegment mirrors af_wire_segment");

namespace {
void wire_free(af_session *s)
{
    s->wr = af_session::Wire{};
    s->wire = s->wire_valid = false;
}

using StreamState = af_session::StreamState;

StreamState fresh_stream(const af_session *s, uint32_t fmt)
{
    StreamState f{};
    f.rec.init(s->fmts[fmt].rate, OUT_RATE);
    f.in_len = 2 * RS_POLY;                                      // rubato starts with 16 zero frames of history
    f.in_base = -2 * RS_POLY;
    f.fmt = fmt;
    return f;
}

uint32_t stream_fmt(const af_session *s, size_t k) { return s->diverged ? s->ss[k].fmt : s->shared.fmt; }
}  // namespace

extern "C" {

AF_API void af_session_destroy(af_session *s)
{
    if (!s) return;
    DevScope scope_(s->device);
    cudaDeviceSynchronize();
    delete s;
}

AF_API int af_session_reset(af_session *s)
{
    if (!s) return fail(AF_ERR_INVALID, "null session");
    AF_SCOPE(s->device);
    // every stream to the common start in its current format: lockstep again when they all share one
    bool one = true;
    for (size_t k = 1; k < s->S && one; ++k) one = stream_fmt(s, k) == stream_fmt(s, 0);
    if (one) {
        s->shared = fresh_stream(s, stream_fmt(s, 0));
        s->diverged = false;
    } else {
        for (size_t k = 0; k < s->S; ++k) s->ss[k] = fresh_stream(s, s->ss[k].fmt);
    }
    s->in_cur = 0; s->y_cur = 0;
    AF_CUDA(cudaMemset(s->in_buf[0].get(), 0, s->S * s->in_stride * sizeof(float)));
    AF_CUDA(cudaMemset(s->d_vad.get(), 0, s->S * sizeof(VadState)));
    if (s->d_wire_prev.get()) AF_CUDA(cudaMemset(s->d_wire_prev.get(), 0, s->S));   // no segment open
    if (s->wr.pre.frames) AF_CUDA(cudaMemset(s->wr.pre.d_n.get(), 0, s->S * sizeof(uint32_t)));   // no pre-roll history
    return AF_OK;
}

AF_API int af_session_create(af_pipeline *p, size_t n_streams, uint32_t sample_rate, uint16_t channels, uint16_t format,
                             uint32_t max_tick_samples, af_session **out)
{
    const af_stream_format f{sample_rate, channels, 0, max_tick_samples};
    return af_session_create_formats(p, n_streams, &f, 1, nullptr, format, out);
}

AF_API int af_session_create_formats(af_pipeline *p, size_t n_streams, const af_stream_format *formats, size_t n_formats,
                                     const uint32_t *stream_format, uint16_t format, af_session **out)
{
    if (!p || !out || n_streams == 0 || (!formats && n_formats)) return fail(AF_ERR_INVALID, "bad argument");
    if (n_formats == 0 || n_formats > (1u << (32 - TICK_FMT_SHIFT)))
        return fail(AF_ERR_INVALID, "%zu formats (a session admits 1 to %u)", n_formats, 1u << (32 - TICK_FMT_SHIFT));
    if (format != AF_FMT_F32 && format != AF_FMT_I16) return fail(AF_ERR_INVALID, "bad stream format");
    for (size_t i = 0; i < n_formats; ++i) {
        const af_stream_format &f = formats[i];
        if (f.channels == 0 || f.sample_rate == 0 || f.max_tick_samples == 0 || f.pad != 0)
            return fail(AF_ERR_INVALID, "bad stream format %zu", i);
    }
    if (stream_format)
        for (size_t k = 0; k < n_streams; ++k)
            if (stream_format[k] >= n_formats)
                return fail(AF_ERR_INVALID, "stream %zu: format %u out of range (%zu formats)", k, stream_format[k], n_formats);
    int rc = require_ctx();
    if (rc) return rc;
    const af_pipeline_config &cfg = p->cfg;
    if (cfg.n_mels && cfg.vad_enable && cfg.vad_frame_len != 0 && (cfg.vad_frame_len != WIN || cfg.vad_hop != HOP))
        return fail(AF_ERR_INVALID, "sessions need the VAD on the STFT frames when features are enabled");
    if (cfg.pcm16) return fail(AF_ERR_INVALID, "sessions deliver f32 PCM (pcm16 is a batch option; af_pcm16_encode converts a tick)");
    std::unique_ptr<af_session, void (*)(af_session *)> s(new af_session, af_session_destroy);
    s->device = cur_device();
    if (p->cfg.n_mels && !(s->d_mel = pipe_mel(p))) return AF_ERR_CUDA;
    s->pipe = p; s->S = n_streams; s->format = format;
    std::vector<SessionFormat> dev(n_formats);
    uint64_t max_new_y = 0;
    for (size_t i = 0; i < n_formats; ++i) {
        const af_stream_format &f = formats[i];
        const uint32_t frames = (f.max_tick_samples + f.channels - 1) / f.channels;
        RsRecurrence rec;
        rec.init(f.sample_rate, OUT_RATE);
        if (!rec.passthrough && rec.end_idx <= 0) return fail(AF_ERR_RESAMPLING_FAILED, "unsupported resampling ratio");
        s->fmts.push_back({f.sample_rate, f.channels, frames});
        dev[i] = {f.channels, rec.p, rec.q, rec.mode()};
        s->any_table = s->any_table || rec.mode() == RS_TABLE;
        s->max_tick_frames = std::max(s->max_tick_frames, frames);
        // (a count of max_samples passes af_session_push_rings_available's check while max_samples / channels <= frames)
        s->max_ring_samples = std::max<uint64_t>(s->max_ring_samples, (uint64_t)f.channels * (frames + 1) - 1);
        max_new_y = std::max<uint64_t>(max_new_y, af_resample_max_output(f.sample_rate, OUT_RATE, frames + RS_CHUNK) + 8);
    }
    s->framing = cfg.n_mels != 0 || cfg.vad_enable;
    if (cfg.vad_enable && cfg.vad_frame_len != 0) { s->frame_len = cfg.vad_frame_len; s->hop = cfg.vad_hop; }
    s->in_stride = round_up(2 * RS_POLY + RS_CHUNK + s->max_tick_frames + 8, 4);
    s->max_new_y = max_new_y;
    s->y_stride = round_up(s->frame_len + s->hop + max_new_y + 8, 4);
    s->packed = s->framing && s->frame_len == WIN && s->hop == HOP;
    if (s->packed) s->y_stride = round_up(s->y_stride, HOP);           // rows a whole number of hops apart (HOP % 4 == 0)
    const uint64_t max_frames = (s->y_stride) / s->hop + 2;
    s->energy_stride = round_up(max_frames, 4);
    s->lm_stride = round_up(max_frames * std::max<uint32_t>(cfg.n_mels, 1), 4);
    if (s->packed) {
        s->pk_slots = (uint32_t)(s->y_stride / HOP);
        s->pk_rows = std::max<uint32_t>(1u, (uint32_t)SF / s->pk_slots);   // about one 32-frame step per virtual stream
        s->pk_n = (uint32_t)((n_streams + s->pk_rows - 1) / s->pk_rows);
        s->energy_stride = s->pk_slots;                                  // frame slot pitch of a real stream
        s->lm_stride = (uint64_t)s->pk_slots * std::max<uint32_t>(cfg.n_mels, 1);
    }
    s->st_stride = round_up(max_frames, 16);
    for (int i = 0; i < 2; ++i) {
        AF_CUDA(s->in_buf[i].alloc(n_streams * s->in_stride));
        AF_CUDA(s->y_buf[i].alloc(n_streams * s->y_stride));
        AF_CUDA(cudaMemset(s->y_buf[i].get(), 0, n_streams * s->y_stride * sizeof(float)));
        if (s->packed) {
            std::vector<StreamDev> ptab(s->pk_n);
            std::vector<TileDev> ptiles(s->pk_n);
            for (uint32_t v = 0; v < s->pk_n; ++v) {
                StreamDev &d = ptab[v];
                memset(&d, 0, sizeof(d));
                const uint64_t rows = std::min<uint64_t>(s->pk_rows, n_streams - (uint64_t)v * s->pk_rows);
                d.data = s->y_buf[i].get() + (uint64_t)v * s->pk_rows * s->y_stride;
                d.n_samples = rows * s->y_stride; d.n_in = d.n_out = (uint32_t)d.n_samples;
                d.n_frames = d.n_vad_frames = 1 + (d.n_out - WIN) / HOP;
                d.channels = 1; d.format = FMT_F32; d.p = 1; d.q = 1; d.mode = RS_PASSTHROUGH;
                d.tile_begin = v; d.n_tiles = 1; d.staged = 2;
                plan_tile(d, v, 0, &ptiles[v]);
            }
            AF_CUDA(s->d_ptab[i].alloc(s->pk_n));
            AF_CUDA(s->d_ptiles[i].alloc(s->pk_n));
            AF_CUDA(cudaMemcpy(s->d_ptab[i].get(), ptab.data(), s->pk_n * sizeof(StreamDev), cudaMemcpyHostToDevice));
            AF_CUDA(cudaMemcpy(s->d_ptiles[i].get(), ptiles.data(), s->pk_n * sizeof(TileDev), cudaMemcpyHostToDevice));
        }
    }
    if (s->y_stride > (uint64_t)TILE_SAMPLES)
        return fail(AF_ERR_INVALID, "max_tick_samples too large for a session (%u frames)", s->max_tick_frames);
    AF_CUDA(s->d_vad.alloc(n_streams));
    AF_CUDA(s->d_energy.alloc(n_streams * s->energy_stride));
    AF_CUDA(s->d_frac.alloc(max_new_y + 64));
    AF_CUDA(s->d_fmts.alloc(n_formats));
    AF_CUDA(cudaMemcpy(s->d_fmts.get(), dev.data(), n_formats * sizeof(SessionFormat), cudaMemcpyHostToDevice));
    s->ss.resize(n_streams); s->ss_next.resize(n_streams);
    for (size_t k = 0; k < n_streams; ++k) s->ss[k].fmt = stream_format ? stream_format[k] : 0;
    s->diverged = true;                            // (af_session_reset reads each stream's format from ss)
    s->first_frames.assign(n_streams, 0);
    rc = af_session_reset(s.get());
    if (rc) return rc;
    *out = s.release();
    return AF_OK;
}

}  // extern "C"

namespace {
bool same_fields(const StreamState &a, const StreamState &b)
{
    return a.fmt == b.fmt && a.rec.chunks == b.rec.chunks && a.rec.n_out == b.rec.n_out &&
           a.rec.last_index == b.rec.last_index && a.in_len == b.in_len && a.in_drop == b.in_drop && a.y_len == b.y_len &&
           a.y_drop == b.y_drop && a.in_base == b.in_base && a.frames_emitted == b.frames_emitted;
}

bool same_position(const StreamState &a, const StreamState &b) { return !a.restart && !b.restart && same_fields(a, b); }

// A stream's plan (its StreamTick, fraction slice and next state) is a function of its format, its position (none while it
// restarts: a fresh stream's), its count and its end flag; streams with equal keys share one plan.
bool same_plan(const StreamState &a, uint32_t na, bool fa, const StreamState &b, uint32_t nb, bool fb)
{
    return na == nb && fa == fb && a.restart == b.restart && (a.restart ? a.fmt == b.fmt : same_fields(a, b));
}

uint64_t plan_hash(const StreamState &a, uint32_t n, bool fin)
{
    uint64_t h = ((uint64_t)a.fmt << 34) ^ ((uint64_t)n << 2) ^ (fin ? 1u : 0u) ^ (a.restart ? 2u : 0u);
    if (!a.restart)
        h ^= a.rec.chunks * 0x9E3779B97F4A7C15ull ^ (uint64_t)a.in_len << 40 ^ (uint64_t)a.y_len * 0xC2B2AE3D27D4EB4Full ^
             (uint64_t)a.in_base * 0x165667B19E3779F9ull ^ a.frames_emitted;
    h ^= h >> 33; h *= 0xFF51AFD7ED558CCDull; h ^= h >> 33;
    return h;
}

// RsRecurrence::step `chunks` times.  An exact recurrence (t = p / q, q a power of two) takes the closed form: the output
// count of rs_exact_count and last_index = -4 + n_out * p / q - 128 * chunks, both exact (the step adds dyadic rationals
// without rounding), so a thousand streams cost no per-output host loop.
void rs_advance(RsRecurrence &r, uint32_t chunks, std::vector<float> *frac)
{
    if (!r.exact) {
        for (uint32_t c = 0; c < chunks; ++c) r.step(frac);
        return;
    }
    if (!chunks) return;
    r.chunks += chunks;
    r.n_out = rs_exact_count(r, r.chunks);
    const long long num = (long long)r.n_out * (long long)r.p - (long long)RS_CHUNK * (long long)r.chunks * (long long)r.q;
    r.last_index = -(double)(RS_POLY / 2) + (double)num / (double)r.q;
}

// one stream's count in a tick: whole frames of its format, at most its format's max_tick_samples, within its input row
int check_count(const af_session *s, uint32_t fmt, uint32_t n, uint64_t in_stride)
{
    const af_session::Format &f = s->fmts[fmt];
    if (n % f.channels) return fail(AF_ERR_INVALID, "a tick of %u samples is not a whole number of frames", n);
    if (n / f.channels > f.max_tick_frames) return fail(AF_ERR_CAPACITY, "tick of %u frames exceeds max_tick_samples", n / f.channels);
    if (in_stride < n) return fail(AF_ERR_INVALID, "in_stride %llu smaller than a tick of %u samples", (unsigned long long)in_stride, n);
    return AF_OK;
}

// Plans one stream's tick of n_samples from its state `now` (a fresh stream when it restarts): fills `d` and the state
// after the tick, `next`, and appends the RS_TABLE fractions to s->frac_host at d.frac_off.  fin ends the stream after
// the tick (BatchResampler::flush, resampler.rs:150-166).  Only internal capacity errors can occur; nothing changes.
int plan_stream(af_session *s, const StreamState &now, uint32_t n_samples, bool fin, StreamTick &d, StreamState &next)
{
    StreamState c = now.restart ? fresh_stream(s, now.fmt) : now;
    // frames held: [history 16 | residual r | new n_new]; chunks formed from residual + new
    const uint32_t n_new = n_samples / s->fmts[c.fmt].channels;
    const uint32_t residual = c.in_len - 2 * RS_POLY;
    const uint32_t avail = residual + n_new;
    const bool pass = c.rec.passthrough;
    const uint32_t full = pass ? 0 : avail / RS_CHUNK;
    // a flush zero-pads a residual to one more chunk.  The bound of max_new_y holds for it: ceil((127 + max_tick_frames)
    // / 128) chunks <= the ceil((max_tick_frames + 128) / 128) it was sized for.
    const uint32_t chunks = full + ((fin && !pass && avail % RS_CHUNK) ? 1 : 0);
    const uint64_t n_begin = pass ? (uint64_t)(c.in_base + 2 * RS_POLY + residual) : c.rec.n_out;
    const size_t frac_off = s->frac_host.size();
    rs_advance(c.rec, chunks, c.rec.mode() == RS_TABLE ? &s->frac_host : nullptr);
    const uint64_t n_end = pass ? n_begin + n_new : c.rec.n_out;
    const uint32_t n_y = (uint32_t)(n_end - n_begin);
    if (c.y_len + n_y > s->y_stride) return fail(AF_ERR_CAPACITY, "internal: 16 kHz carry overflow");
    const uint32_t y_total = c.y_len + n_y;
    uint32_t T = 0;
    if (s->framing && y_total >= s->frame_len) T = 1 + (y_total - s->frame_len) / s->hop;
    if (T && s->packed && T + 2 > s->pk_slots) return fail(AF_ERR_CAPACITY, "internal: %u frames do not fit %u frame slots", T, s->pk_slots);
    d.in_drop = c.in_drop; d.in_keep = c.in_len; d.n_new = n_new; d.n_samples = n_samples;
    d.data_base = c.in_base;
    d.n_valid_end = pass ? c.in_base + (long long)(c.in_len + n_new)
                         : c.in_base + 2 * RS_POLY + (long long)(fin ? avail : full * RS_CHUNK);
    d.n_begin = n_begin; d.n_y = n_y; d.frac_off = (uint32_t)frac_off;
    d.y_drop = c.y_drop; d.y_keep = c.y_len;
    d.T = T; d.flags = (now.restart ? TICK_RESTART : 0u) | (fin ? TICK_END : 0u) | (c.fmt << TICK_FMT_SHIFT);
    // the consumed chunks and the samples every future frame starts after are dropped by the next tick's ingest /
    // resample (in_drop, y_drop): no kernel and no second synchronisation
    c.in_len += n_new;
    if (!pass) {
        const uint32_t consumed = full * RS_CHUNK;              // keep [history 16 | new residual]
        c.in_drop = consumed; c.in_len -= consumed; c.in_base += consumed;
    } else {
        // passthrough keeps nothing but the 16-frame history slot
        c.in_drop = c.in_len - 2 * RS_POLY; c.in_base += (long long)(c.in_len - 2 * RS_POLY); c.in_len = 2 * RS_POLY;
    }
    const uint32_t y_drop = s->framing ? std::min(T * s->hop, y_total) : y_total;
    c.y_drop = y_drop; c.y_len = y_total - y_drop;
    c.frames_emitted += T;
    c.restart = fin;
    next = c;
    return AF_OK;
}

// One tick.  per_stream: stream k pushes n_samples[k] from its own position ss[k] (end[k] != 0: its last tick), planned
// into the uploaded table h_tick / d_tick that af_session_tick_streams_kernel reads.  Otherwise every stream pushes
// n_samples[0] from `shared`, and af_session_tick_kernel takes that one plan as kernel parameters.  Everything after the
// tick kernel is the same code for both.  Argument errors are reported before anything changes; the bookkeeping is
// committed after the tick's synchronise, so an AF_ERR_CUDA leaves it as it was (reset after one: the detector and wire
// state on the device may have advanced, and af_session_wire refuses the rows until the next push).
int session_tick(af_session *s, const void *data, uint64_t in_stride, const uint32_t *n_samples, const uint8_t *end,
                 bool per_stream, int mem, const af_outputs *o, uint32_t *n_pcm, uint32_t *n_feat, uint32_t *n_vad)
{
    AF_SCOPE(s->device);
    const af_pipeline_config &cfg = s->pipe->cfg;
    cudaStream_t st = cur_ctx().stream;
    const size_t S = s->S;
    const uint32_t bps = s->format == AF_FMT_I16 ? 2 : 4;
    af_outputs none{};
    if (!o) o = &none;

    // ---- 0. plan every stream on copies of its state; validate every caller-supplied size ----
    StreamTick one{};                   // the lockstep plan (all zero on a per-stream tick, whose kernels read the table)
    StreamState shared_next{};
    s->frac_host.clear();               // (scratch, not state)
    uint32_t maxT = 0, max_ny = 0, max_n = 0;
    const size_t tick_bytes = S * (sizeof(StreamTick) + sizeof(uint32_t));
    // the fractions of every distinct plan, one slice after another (a lockstep tick has one)
    AF_CUDA(s->d_frac.grow(per_stream && s->any_table ? S * s->max_new_y : s->max_new_y + 64));
    if (!per_stream) {
        const int rc = plan_stream(s, s->shared, n_samples[0], false, one, shared_next);
        if (rc) return rc;
        maxT = one.T; max_ny = one.n_y; max_n = n_samples[0];
    } else {
        if (!s->tick.d.get()) {                                  // set together: a failed allocation leaves neither
            af_session::TickPlan t;
            const size_t n = (tick_bytes + sizeof(StreamTick) - 1) / sizeof(StreamTick);
            cudaError_t e = t.d.alloc(n);
            if (e == cudaSuccess) e = t.h.alloc(n);
            if (e != cudaSuccess) return fail(AF_ERR_CUDA, "allocating the tick plan: %s", cudaGetErrorString(e));
            s->tick = std::move(t);
        }
        if (!s->diverged) s->ss.assign(S, s->shared);
        StreamTick *h_tick = s->tick.h.get();
        uint32_t *Ts = reinterpret_cast<uint32_t *>(h_tick + S);
        size_t cap = 1;
        while (cap < 2 * S) cap <<= 1;
        s->plan_slots.assign(cap, UINT32_MAX);              // stream that planned each distinct key first
        for (size_t k = 0; k < S; ++k) {
            const bool fin = end && end[k];
            size_t i = plan_hash(s->ss[k], n_samples[k], fin) & (cap - 1);
            for (uint32_t j; (j = s->plan_slots[i]) != UINT32_MAX; i = (i + 1) & (cap - 1))
                if (same_plan(s->ss[j], n_samples[j], end && end[j], s->ss[k], n_samples[k], fin)) break;
            if (s->plan_slots[i] == UINT32_MAX) {
                s->plan_slots[i] = (uint32_t)k;
                const int rc = plan_stream(s, s->ss[k], n_samples[k], fin, h_tick[k], s->ss_next[k]);
                if (rc) return rc;
            } else {                                             // the same plan, and the same fraction slice
                h_tick[k] = h_tick[s->plan_slots[i]];
                s->ss_next[k] = s->ss_next[s->plan_slots[i]];
            }
            Ts[k] = h_tick[k].T;
            maxT = std::max(maxT, Ts[k]); max_ny = std::max(max_ny, h_tick[k].n_y); max_n = std::max(max_n, n_samples[k]);
        }
    }
    if (s->frac_host.size() > s->d_frac.size()) return fail(AF_ERR_CAPACITY, "internal: fraction buffer overflow");
    const bool want_pcm = cfg.write_pcm && o->pcm && max_ny;
    const bool want_lm = maxT && cfg.n_mels && o->logmel;
    const bool want_states = maxT && cfg.vad_enable && o->vad;
    // the wire output needs the tick's states for its events and its gate, whatever the caller asked for; its features
    // need the tick's log-mel the same way
    const bool need_states = want_states || (s->wire && maxT && cfg.vad_enable);
    const bool feats = s->wire && s->wr.feat.d_rows.get();
    const bool need_lm = want_lm || (feats && maxT);
    if (want_pcm && o->pcm_stride < max_ny) return fail(AF_ERR_CAPACITY, "pcm_stride %llu too small for %u samples", (unsigned long long)o->pcm_stride, max_ny);
    if (want_lm && o->logmel_stride < (uint64_t)maxT * cfg.n_mels) return fail(AF_ERR_CAPACITY, "logmel_stride too small for %u frames", maxT);
    if (want_states && o->vad_stride < maxT) return fail(AF_ERR_CAPACITY, "vad_stride too small for %u frames", maxT);
    // internal staging buffers (allocation failures are reported before anything changes, too)
    float *lm = nullptr; uint64_t lm_stride = 0;
    uint8_t *states = nullptr; uint64_t st_stride = 0;
    if (need_lm) {
        if (mem == AF_MEM_HOST || s->packed || !want_lm) {      // (packed ticks write every frame slot: internal buffer, then a strided copy)
            AF_CUDA(s->d_lm.grow(S * s->lm_stride));
            lm = s->d_lm.get(); lm_stride = s->lm_stride;
        } else { lm = o->logmel; lm_stride = o->logmel_stride; }
        if (lm_stride < (uint64_t)maxT * cfg.n_mels) return fail(AF_ERR_CAPACITY, "internal: log-mel staging too small for %u frames", maxT);
    }
    if (need_states) {
        if (mem == AF_MEM_HOST || !want_states) {
            AF_CUDA(s->d_states.grow(S * s->st_stride));
            states = s->d_states.get(); st_stride = s->st_stride;
        } else { states = o->vad; st_stride = o->vad_stride; }
        if (st_stride < maxT) return fail(AF_ERR_CAPACITY, "internal: state staging too small for %u frames", maxT);
    }
    // bound of this tick's payloads: gated, the tick's frames and, once one completed, the pre-roll of earlier pushes
    const uint32_t pre = s->wire ? s->wr.pre.frames : 0;
    const uint64_t wire_n = s->wr.cfg.gate ? (uint64_t)(maxT ? maxT + pre : 0) * s->hop : max_ny;
    if (s->wire && wire_n > s->wr.cap) return fail(AF_ERR_CAPACITY, "internal: %llu wire samples exceed the rows", (unsigned long long)wire_n);
    float *pcm_rows = nullptr; uint64_t pcm_rows_stride = 0;   // per-stream: the tick kernel writes each stream's PCM here
    if (want_pcm && per_stream) {
        if (mem == AF_MEM_HOST) {
            const uint64_t w = round_up(s->max_new_y, 4);
            AF_CUDA(s->d_pcm_stage.grow(S * w));
            pcm_rows = s->d_pcm_stage.get(); pcm_rows_stride = w;
        } else { pcm_rows = o->pcm; pcm_rows_stride = o->pcm_stride; }
    }
    const void *d_in = data;
    uint64_t d_in_stride_bytes = in_stride * bps;
    if (mem == AF_MEM_HOST && max_n) {
        const size_t row = round_up((uint64_t)max_n * bps, 16);
        AF_CUDA(s->d_in_stage.grow(row * S));
        d_in = s->d_in_stage.get(); d_in_stride_bytes = row;
    }

    // From here on only CUDA failures can occur.
    s->wire_valid = false;
    // ---- 1. input: host rows are staged (the caller's buffer may end after the last row's own count: unless that is
    //         the largest, the last row is copied on its own); then the plan and the tick kernel ----
    if (mem == AF_MEM_HOST && max_n) {
        const uint32_t n_last = per_stream ? n_samples[S - 1] : max_n;
        const size_t rows = n_last == max_n ? S : S - 1;
        AF_CUDA(cudaMemcpy2DAsync(s->d_in_stage.get(), d_in_stride_bytes, data, in_stride * bps, (size_t)max_n * bps, rows,
                                  cudaMemcpyHostToDevice, st));
        if (rows < S && n_last)
            AF_CUDA(cudaMemcpyAsync(s->d_in_stage.get() + (S - 1) * d_in_stride_bytes,
                                    static_cast<const char *>(data) + (S - 1) * in_stride * bps, (size_t)n_last * bps,
                                    cudaMemcpyHostToDevice, st));
    }
    if (per_stream) AF_CUDA(cudaMemcpyAsync(s->tick.d.get(), s->tick.h.get(), tick_bytes, cudaMemcpyHostToDevice, st));
    if (!s->frac_host.empty())
        AF_CUDA(cudaMemcpyAsync(s->d_frac.get(), s->frac_host.data(), s->frac_host.size() * sizeof(float), cudaMemcpyHostToDevice, st));
    const int in_next = s->in_cur ^ 1, y_next = s->y_cur ^ 1;
    const StreamTick *tab = per_stream ? s->tick.d.get() : nullptr;
    const uint32_t *d_T = per_stream ? reinterpret_cast<const uint32_t *>(tab + S) : nullptr;
    SessionIngest ing{};
    ing.old_buf = s->in_buf[s->in_cur].get(); ing.new_buf = s->in_buf[in_next].get(); ing.buf_stride = s->in_stride;
    ing.input = d_in; ing.in_stride_bytes = d_in_stride_bytes; ing.channels = s->fmts[s->shared.fmt].channels;
    ing.format = s->format;
    SessionResample rs{};
    rs.in_buf = s->in_buf[in_next].get(); rs.in_stride = s->in_stride;
    rs.p = s->shared.rec.p; rs.q = s->shared.rec.q; rs.mode = s->shared.rec.mode(); rs.frac = s->d_frac.get();
    rs.y_old = s->y_buf[s->y_cur].get(); rs.y_new = s->y_buf[y_next].get(); rs.y_stride = s->y_stride;
    if (per_stream) {
        AF_CUDA(launch_session_tick_streams(ing, rs, tab, s->d_fmts.get(), s->d_vad.get(), s->d_wire_prev.get(), pcm_rows, pcm_rows_stride, (uint32_t)S, st));
    } else {                                                     // the fields the streams kernel takes from its descriptor
        ing.drop = one.in_drop; ing.keep = one.in_keep; ing.n_samples = one.n_samples; ing.n_new_frames = one.n_new;
        rs.data_base = one.data_base; rs.n_valid_end = one.n_valid_end; rs.n_begin = one.n_begin; rs.n_end = one.n_begin + one.n_y;
        rs.y_drop = one.y_drop; rs.y_keep = one.y_keep;
        AF_CUDA(launch_session_tick(ing, rs, (uint32_t)S, st));
    }
    count_launch();
    float *ycur = s->y_buf[y_next].get();

    // ---- 2. PCM (lockstep: copied out of the 16 kHz rows; per-stream: written by the tick kernel), levels ----
    if (want_pcm && !per_stream)
        AF_CUDA(cudaMemcpy2DAsync(o->pcm, o->pcm_stride * sizeof(float), ycur + one.y_keep, s->y_stride * sizeof(float),
                                  (size_t)max_ny * sizeof(float), S,
                                  mem == AF_MEM_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice, st));
    else if (want_pcm && mem == AF_MEM_HOST)
        AF_CUDA(cudaMemcpy2DAsync(o->pcm, o->pcm_stride * sizeof(float), pcm_rows, pcm_rows_stride * sizeof(float),
                                  (size_t)max_ny * sizeof(float), S, cudaMemcpyDeviceToHost, st));
    if (s->levels) {
        AF_CUDA(launch_peak(ycur + one.y_keep, s->y_stride, one.n_y, (uint32_t)S, s->lv.d_peak.get(), st, tab));
        count_launch();
    }

    // ---- 3. frames that became complete: features + VAD.  STFT frames with framing are always packed: the packed
    //         launch computes every frame slot of every row; the energies of custom frames and the scan take each
    //         stream's count ----
    if (maxT) {
        if (s->packed) {
            FusedParams P{};
            P.streams = s->d_ptab[y_next].get(); P.tiles = s->d_ptiles[y_next].get(); P.n_tiles = s->pk_n;
            const uint64_t vrows = s->pk_rows;                  // real streams per stream of the launch
            P.fft = cur_ctx().d_fft.get(); P.mel = s->d_mel;
            P.pcm = nullptr; P.pcm_stride = 0;
            P.logmel = lm; P.logmel_stride = lm_stride * vrows;
            P.energy = cfg.vad_enable ? s->d_energy.get() : nullptr; P.energy_stride = s->energy_stride * vrows;
            P.n_mels = lm ? cfg.n_mels : 0;
            P.do_energy = cfg.vad_enable ? 1 : 0;
            P.log_floor = cfg.log_floor;
            P.log_scale = cfg.log10 ? 0.30102999566398120f : 0.69314718055994531f;
            P.use_stage = kernel_variant() == "sync" ? 0u : 1u;
            P.layout = fused_layout(P.do_energy != 0);
            P.neg_zero = -0.0f;
            if (P.n_mels || P.do_energy) {
                AF_CUDA(launch_fused(P, (int)std::min<size_t>(P.n_tiles, (size_t)cur_ctx().sm_count), st));
                count_launch(2);
            }
        } else {
            EnergyJob ej{};
            ej.y = ycur; ej.y_stride = s->y_stride; ej.n_frames = d_T; ej.n_frames_all = maxT;
            ej.frame_len = s->frame_len; ej.hop = s->hop; ej.energy = s->d_energy.get(); ej.energy_stride = s->energy_stride;
            ej.n_streams = (uint32_t)S;
            AF_CUDA(launch_frame_energy(ej, st));
            count_launch();
        }
        if (cfg.vad_enable) {
            ScanJob sj{};
            sj.energy = s->d_energy.get(); sj.energy_stride = s->energy_stride; sj.n_frames = d_T; sj.n_frames_all = maxT;
            sj.states = states; sj.states_stride = st_stride; sj.state_io = s->d_vad.get();
            sj.final_out = mem == AF_MEM_DEVICE ? reinterpret_cast<VadState *>(o->vad_final) : nullptr;
            sj.prm = s->pipe->vad_prm; sj.n_streams = (uint32_t)S;
            if (s->n_custom_recs) {                              // the records set since the last upload, in one copy
                if (s->recs_lo < s->recs_hi)
                    AF_CUDA(cudaMemcpyAsync(s->d_recs.get() + s->recs_lo, s->h_recs.get() + s->recs_lo,
                                            (s->recs_hi - s->recs_lo) * sizeof(ScanRec), cudaMemcpyHostToDevice, st));
                s->recs_lo = S; s->recs_hi = 0;
                sj.recs = s->d_recs.get();
            }
            AF_CUDA(launch_vad_scan(sj, st));
            count_launch();
        }
        if (mem == AF_MEM_DEVICE && want_lm && lm != o->logmel)
            AF_CUDA(cudaMemcpy2DAsync(o->logmel, o->logmel_stride * sizeof(float), lm, lm_stride * sizeof(float),
                                      (size_t)maxT * cfg.n_mels * sizeof(float), S, cudaMemcpyDeviceToDevice, st));
        if (mem == AF_MEM_HOST) {
            if (want_lm) AF_CUDA(cudaMemcpy2DAsync(o->logmel, o->logmel_stride * sizeof(float), lm, lm_stride * sizeof(float),
                                              (size_t)maxT * cfg.n_mels * sizeof(float), S, cudaMemcpyDeviceToHost, st));
            if (want_states) AF_CUDA(cudaMemcpy2DAsync(o->vad, o->vad_stride, states, st_stride, maxT, S, cudaMemcpyDeviceToHost, st));
        }
    }
    // every stream's detector (a restarted one is fresh), whether or not a frame completed; the scan wrote device rows
    if (cfg.vad_enable && o->vad_final && (mem == AF_MEM_HOST || !maxT))
        AF_CUDA(cudaMemcpyAsync(o->vad_final, s->d_vad.get(), S * sizeof(VadState),
                                mem == AF_MEM_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice, st));
    // ---- 4. wire payloads: one launch for all streams after the scan; host rows receive only what bounds the payloads ----
    if (s->wire) {
        const af_session::Wire &wr = s->wr;
        const af_session::Wire::Segments &ws = wr.seg;
        if (feats && !pre) {                                     // before the wire kernel, which advances d_wire_prev
            const af_session::Wire::Features &wf = wr.feat;
            WireLogmelJob fj{};
            fj.lm = lm; fj.lm_stride = lm_stride; fj.n_mels = cfg.n_mels;
            fj.states = maxT ? states : nullptr; fj.st_stride = st_stride; fj.T = maxT;
            fj.prev = s->d_wire_prev.get();
            fj.out = wf.d_rows.get(); fj.out_stride = wf.stride; fj.n_frames = wf.d_n.get();
            fj.n_streams = (uint32_t)S; fj.tab = tab;
            AF_CUDA(launch_session_wire_logmel(fj, st));
            count_launch();
            // (the rows hold the wire's bound of frames, and wire_n <= wr.cap above bounds maxT by it)
            if (wf.mem == AF_MEM_HOST && maxT)
                AF_CUDA(cudaMemcpy2DAsync(wf.h_rows.get(), wf.stride * sizeof(float), wf.d_rows.get(), wf.stride * sizeof(float),
                                          (size_t)maxT * cfg.n_mels * sizeof(float), S, cudaMemcpyDeviceToHost, st));
            AF_CUDA(cudaMemcpyAsync(wf.h_n.get(), wf.d_n.get(), S * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        }
        if (pre) {                                               // one launch: payloads, features, records, history
            const af_session::Wire::Features &wf = wr.feat;
            WirePrerollJob pj{};
            pj.y = ycur; pj.y_stride = s->y_stride;
            pj.states = maxT ? states : nullptr; pj.st_stride = st_stride;
            pj.T = maxT; pj.hop = s->hop; pj.P = pre;
            pj.prev = s->d_wire_prev.get();
            pj.pcm16 = wr.d_pcm16.get(); pj.pcm16_stride = wr.pcm16_stride;
            pj.b64 = wr.d_b64.get(); pj.b64_stride = wr.b64_stride;
            pj.ticks = wr.d_ticks.get();
            if (feats) {
                pj.lm = lm; pj.lm_stride = lm_stride; pj.n_mels = cfg.n_mels;
                pj.lm_out = wf.d_rows.get(); pj.lm_out_stride = wf.stride; pj.n_frames = wf.d_n.get();
                pj.hist_lm = wr.pre.d_lm.get();
            }
            pj.hist_pcm = wr.pre.d_pcm.get(); pj.hist_n = wr.pre.d_n.get(); pj.hist_pos = wr.pre.d_pos.get();
            pj.n_streams = (uint32_t)S; pj.tab = tab;
            pj.segs = ws.d_rows.get(); pj.seg_stride = ws.stride; pj.n_segs = ws.d_n.get();
            AF_CUDA(launch_session_wire_preroll(pj, st));
            count_launch();
            if (feats) {
                if (wf.mem == AF_MEM_HOST && wire_n)
                    AF_CUDA(cudaMemcpy2DAsync(wf.h_rows.get(), wf.stride * sizeof(float), wf.d_rows.get(), wf.stride * sizeof(float),
                                              (size_t)(wire_n / s->hop) * cfg.n_mels * sizeof(float), S, cudaMemcpyDeviceToHost, st));
                AF_CUDA(cudaMemcpyAsync(wf.h_n.get(), wf.d_n.get(), S * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
            }
        } else {
            WireJob wj{};
            wj.y = ycur; wj.y_stride = s->y_stride; wj.y_new = one.y_keep; wj.n_new = one.n_y;
            wj.states = (maxT && cfg.vad_enable) ? states : nullptr; wj.st_stride = st_stride;
            wj.T = maxT; wj.hop = s->hop; wj.gate = wr.cfg.gate;          // (T sizes the kept-frame list: the largest)
            wj.prev = s->d_wire_prev.get();
            wj.pcm16 = wr.d_pcm16.get(); wj.pcm16_stride = wr.pcm16_stride;
            wj.b64 = wr.d_b64.get(); wj.b64_stride = wr.b64_stride;
            wj.ticks = wr.d_ticks.get(); wj.n_streams = (uint32_t)S; wj.tab = tab;
            wj.segs = ws.d_rows.get(); wj.seg_stride = ws.stride; wj.n_segs = ws.d_n.get();
            AF_CUDA(launch_session_wire(wj, st));
            count_launch();
        }
        if (ws.d_rows.get()) {                                   // (a tick of T frames has at most ceil(T / 2) + 1 pieces)
            if (ws.mem == AF_MEM_HOST)
                AF_CUDA(cudaMemcpy2DAsync(ws.h_rows.get(), ws.stride * sizeof(WireSegment), ws.d_rows.get(),
                                          ws.stride * sizeof(WireSegment), ((maxT + 1) / 2 + 1) * sizeof(WireSegment), S,
                                          cudaMemcpyDeviceToHost, st));
            AF_CUDA(cudaMemcpyAsync(ws.h_n.get(), ws.d_n.get(), S * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        }
        if (wr.cfg.mem == AF_MEM_HOST && wire_n) {
            if (wr.cfg.pcm16)
                AF_CUDA(cudaMemcpy2DAsync(wr.h_pcm16.get(), wr.pcm16_stride * sizeof(int16_t), wr.d_pcm16.get(),
                                          wr.pcm16_stride * sizeof(int16_t), wire_n * sizeof(int16_t), S, cudaMemcpyDeviceToHost, st));
            if (wr.cfg.base64)
                AF_CUDA(cudaMemcpy2DAsync(wr.h_b64.get(), wr.b64_stride, wr.d_b64.get(), wr.b64_stride,
                                          af_pcm16_base64_len(wire_n), S, cudaMemcpyDeviceToHost, st));
        }
        AF_CUDA(cudaMemcpyAsync(wr.h_ticks.get(), wr.d_ticks.get(), S * sizeof(af_wire_tick), cudaMemcpyDeviceToHost, st));
    }
    if (s->levels) {
        AF_CUDA(cudaMemcpyAsync(s->lv.h_peak.get(), s->lv.d_peak.get(), S * sizeof(float), cudaMemcpyDeviceToHost, st));
        AF_CUDA(cudaMemcpyAsync(s->lv.h_vad.get(), s->d_vad.get(), S * sizeof(VadState), cudaMemcpyDeviceToHost, st));
    }
    AF_CUDA(cudaStreamSynchronize(st));

    // ---- 5. commit; streams that all stand at the same position run in lockstep again ----
    s->in_cur = in_next; s->y_cur = y_next;
    s->levels_valid = s->levels;
    s->wire_valid = s->wire;
    if (feats) s->wr.feat.valid = true;
    if (s->wire && s->wr.seg.d_rows.get()) s->wr.seg.valid = true;
    if (!per_stream) {
        s->shared = shared_next;
    } else {
        s->ss.swap(s->ss_next);
        bool aligned = true;
        for (size_t k = 0; k < S && aligned; ++k) aligned = same_position(s->ss[k], s->ss[0]);
        s->diverged = !aligned;
        if (aligned) s->shared = s->ss[0];
    }
    for (size_t k = 0; k < S; ++k) {
        const StreamTick &d = per_stream ? s->tick.h.get()[k] : one;
        s->first_frames[k] = (per_stream ? s->ss[k] : s->shared).frames_emitted - d.T;
        if (n_pcm) n_pcm[k] = d.n_y;
        if (n_feat) n_feat[k] = cfg.n_mels ? d.T : 0;
        if (n_vad) n_vad[k] = cfg.vad_enable ? d.T : 0;
    }
    return AF_OK;
}

// The per-stream configuration tables, allocated once: every slot starts with the pipeline's (both tables or neither;
// the first upload takes all)
int alloc_vad_configs(af_session *s)
{
    if (s->h_recs.get()) return AF_OK;
    PinnedBuf<ScanRec> h;
    DevBuf<ScanRec> d;
    AF_CUDA(h.alloc(s->S));
    AF_CUDA(d.alloc(s->S));
    std::fill(h.get(), h.get() + s->S, scan_rec(s->pipe->vad_prm));
    s->h_recs = std::move(h);
    s->d_recs = std::move(d);
    s->vad_cfgs.assign(s->S, s->pipe->cfg.vad);
    s->recs_lo = 0; s->recs_hi = s->S;
    return AF_OK;
}

// Stream streams[i] takes cfgs[i], in order (the last entry for a stream wins); the tables exist
void put_vad_configs(af_session *s, const uint32_t *streams, const af_vad_config *cfgs, size_t n)
{
    const ScanRec base = scan_rec(s->pipe->vad_prm);
    std::vector<ScanRec> recs(n);
    make_scan_recs(cfgs, n, recs.data());
    ScanRec *h = s->h_recs.get();
    for (size_t i = 0; i < n; ++i) {
        const uint32_t k = streams[i];
        s->n_custom_recs -= same_rec(h[k], base) ? 0 : 1;
        h[k] = recs[i];
        s->vad_cfgs[k] = cfgs[i];
        s->n_custom_recs += same_rec(h[k], base) ? 0 : 1;
        s->recs_lo = std::min<size_t>(s->recs_lo, k);
        s->recs_hi = std::max<size_t>(s->recs_hi, (size_t)k + 1);
    }
}
}  // namespace

extern "C" {

AF_API int af_session_push(af_session *s, const void *data, uint64_t in_stride, uint32_t n_samples, int mem,
                           const af_outputs *o, uint32_t *n_pcm, uint32_t *n_feat, uint32_t *n_vad)
{
    if (!s || (!data && n_samples)) return fail(AF_ERR_INVALID, "null argument");
    if (s->diverged) {                                           // streams on their own timelines: the same count for each
        s->counts.assign(s->S, n_samples);
        return af_session_push_streams(s, data, in_stride, s->counts.data(), nullptr, mem, o, n_pcm, n_feat, n_vad);
    }
    if (mem != AF_MEM_DEVICE && mem != AF_MEM_HOST) return fail(AF_ERR_INVALID, "bad memory kind %d", mem);
    const int rc = check_count(s, s->shared.fmt, n_samples, in_stride);
    if (rc) return rc;
    return session_tick(s, data, in_stride, &n_samples, nullptr, false, mem, o, n_pcm, n_feat, n_vad);
}

AF_API int af_session_push_streams(af_session *s, const void *data, uint64_t in_stride, const uint32_t *n_samples,
                                   const uint8_t *end, int mem, const af_outputs *out,
                                   uint32_t *n_pcm, uint32_t *n_feat, uint32_t *n_vad)
{
    if (!s || !n_samples) return fail(AF_ERR_INVALID, "null argument");
    if (mem != AF_MEM_DEVICE && mem != AF_MEM_HOST) return fail(AF_ERR_INVALID, "bad memory kind %d", mem);
    bool equal = true, any_end = false;
    for (size_t k = 0; k < s->S; ++k) {
        const uint32_t n = n_samples[k];
        const int rc = check_count(s, stream_fmt(s, k), n, in_stride);
        if (rc) return rc;
        if (n && !data) return fail(AF_ERR_INVALID, "null data");
        equal = equal && n == n_samples[0];
        any_end = any_end || (end && end[k]);
    }
    // every stream at the shared position and the same count: the lockstep tick (same launches and copies as always)
    return session_tick(s, data, in_stride, n_samples, end, s->diverged || !equal || any_end, mem, out, n_pcm, n_feat, n_vad);
}

AF_API int af_session_reset_streams(af_session *s, const uint32_t *streams, size_t n)
{
    if (!s || (!streams && n)) return fail(AF_ERR_INVALID, "null argument");
    for (size_t i = 0; i < n; ++i)
        if (streams[i] >= s->S) return fail(AF_ERR_INVALID, "stream index %u out of range (%zu streams)", streams[i], s->S);
    if (!n) return AF_OK;
    if (!s->diverged) {
        s->ss.assign(s->S, s->shared);
        s->diverged = true;
    }
    for (size_t i = 0; i < n; ++i) s->ss[streams[i]].restart = true;   // applied by the stream's next tick kernel
    return AF_OK;
}

AF_API int af_session_restart_streams(af_session *s, const uint32_t *streams, const uint32_t *format, size_t n)
{
    if (!s || ((!streams || !format) && n)) return fail(AF_ERR_INVALID, "null argument");
    for (size_t i = 0; i < n; ++i) {
        if (streams[i] >= s->S) return fail(AF_ERR_INVALID, "stream index %u out of range (%zu streams)", streams[i], s->S);
        if (format[i] >= s->fmts.size()) return fail(AF_ERR_INVALID, "format index %u out of range (%zu formats)", format[i], s->fmts.size());
    }
    const int rc = af_session_reset_streams(s, streams, n);
    if (rc) return rc;
    for (size_t i = 0; i < n; ++i) s->ss[streams[i]].fmt = format[i];   // the format of the next life
    return AF_OK;
}

AF_API int af_session_set_vad_configs(af_session *s, const uint32_t *streams, const af_vad_config *cfgs, size_t n)
{
    if (!s || ((!streams || !cfgs) && n)) return fail(AF_ERR_INVALID, "null argument");
    if (!s->pipe->cfg.vad_enable) return fail(AF_ERR_INVALID, "the pipeline runs no VAD (vad_enable == 0)");
    for (size_t i = 0; i < n; ++i)
        if (streams[i] >= s->S) return fail(AF_ERR_INVALID, "stream index %u out of range (%zu streams)", streams[i], s->S);
    if (!n) return AF_OK;
    AF_SCOPE(s->device);
    const int rc = alloc_vad_configs(s);
    if (rc) return rc;
    put_vad_configs(s, streams, cfgs, n);
    return AF_OK;
}

AF_API int af_session_wire_first_frames(const af_session *s, uint64_t *first_frame)
{
    if (!s || !first_frame) return fail(AF_ERR_INVALID, "null argument");
    if (!s->wire_valid) return fail(AF_ERR_INVALID, "no tick has been pushed since af_session_enable_wire");
    std::copy(s->first_frames.begin(), s->first_frames.end(), first_frame);
    return AF_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------
// stream records: a live stream's complete state as bytes, continued by any compatible session on any GPU
// ------------------------------------------------------------------------------------------
namespace {
constexpr uint32_t REC_MAGIC = 0x53524641u;               // "AFRS"
constexpr uint32_t REC_VERSION = 1;                       // bump with any change of the layout or of what a field means
constexpr uint32_t REC_FRAMING = 1, REC_VAD = 2, REC_RESTART = 4, REC_WIRE = 8;

// The host-written head of a record; RecordDev and the two float ranges follow (af_launch.h).  The position is copied
// field by field, never recomputed: on table-mode rates the f64 last_index drifts from the closed form, and every later
// output's fraction depends on its exact bits.
struct StreamRecord {
    uint32_t magic, version, bytes;
    uint32_t frame_len, hop, flags;                       // framing (REC_FRAMING, REC_VAD) and state (REC_RESTART, REC_WIRE)
    uint32_t rate, channels;
    uint64_t last_index;                                  // RsRecurrence::last_index, the f64 bit pattern
    uint64_t chunks, n_out;                               // RsRecurrence::chunks, n_out
    int64_t in_base;
    uint64_t frames_emitted;
    uint32_t in_len, y_len;                               // the two ranges (0, 0 for a pending restart)
    af_vad_config vad;                                    // the stream's effective configuration
    uint32_t pad[2];                                      // 0
};
static_assert(sizeof(StreamRecord) % 16 == 0 && sizeof(RecordDev) == 32, "record parts keep 16-byte alignment");

uint32_t framing_flags(const af_session *s)
{
    return (s->framing ? REC_FRAMING : 0u) | (s->pipe->cfg.vad_enable ? REC_VAD : 0u);
}

size_t record_bytes(const af_session *s)
{
    return round_up(sizeof(StreamRecord) + sizeof(RecordDev) + sizeof(float) * (REC_IN_FRAMES + s->frame_len), 16);
}

// the move table in pinned memory, its device copy, and (n_hdr records) the pinned headers of device records
int reserve_transfer(af_session *s, size_t n, size_t n_hdr)
{
    af_session::Transfer &x = s->xfer;
    if (n > x.h_moves.size() || n > x.d_moves.size()) {
        AF_CUDA(x.h_moves.alloc(n));
        AF_CUDA(x.d_moves.alloc(n));
    }
    AF_CUDA(x.h_hdr.grow(n_hdr * sizeof(StreamRecord)));
    return AF_OK;
}

RecordJob record_job(af_session *s, uint8_t *rec)
{
    RecordJob j{};
    j.tab = s->xfer.d_moves.get();
    j.rec = rec; j.rec_bytes = record_bytes(s); j.dev_off = sizeof(StreamRecord);
    j.n_floats = (uint32_t)((j.rec_bytes - sizeof(StreamRecord) - sizeof(RecordDev)) / sizeof(float));
    j.in_buf = s->in_buf[s->in_cur].get(); j.in_stride = s->in_stride;
    j.y_buf = s->y_buf[s->y_cur].get(); j.y_stride = s->y_stride;
    j.vad = s->d_vad.get();
    j.wire_prev = s->d_wire_prev.get();
    return j;
}

// A record's header against this session: AF_OK and the format it lands in, or AF_ERR_INVALID
int check_record(const af_session *s, const StreamRecord &r, size_t i, const uint32_t *format, uint32_t *fmt)
{
    if (r.magic != REC_MAGIC || r.version != REC_VERSION)
        return fail(AF_ERR_INVALID, "record %zu: not a stream record of this library build", i);
    if (r.bytes != record_bytes(s)) return fail(AF_ERR_INVALID, "record %zu: %u bytes, this session's are %zu", i, r.bytes, record_bytes(s));
    if ((r.flags & (REC_FRAMING | REC_VAD)) != framing_flags(s) || r.frame_len != s->frame_len || r.hop != s->hop)
        return fail(AF_ERR_INVALID, "record %zu: framing %u/%u (flags %u) differs from this session's %u/%u (flags %u)", i,
                    r.frame_len, r.hop, r.flags & (REC_FRAMING | REC_VAD), s->frame_len, s->hop, framing_flags(s));
    if (r.in_len > REC_IN_FRAMES || (r.flags & REC_FRAMING ? r.y_len >= s->frame_len : r.y_len != 0))
        return fail(AF_ERR_INVALID, "record %zu: corrupted ranges", i);
    if (format) {
        if (format[i] >= s->fmts.size()) return fail(AF_ERR_INVALID, "record %zu: format index %u out of range (%zu formats)", i, format[i], s->fmts.size());
        const af_session::Format &f = s->fmts[format[i]];
        if (f.rate != r.rate || f.channels != r.channels)
            return fail(AF_ERR_INVALID, "record %zu: format %u is %u Hz x %u, the record's stream %u Hz x %u", i, format[i], f.rate,
                        f.channels, r.rate, r.channels);
        *fmt = format[i];
        return AF_OK;
    }
    for (uint32_t k = 0; k < s->fmts.size(); ++k)
        if (s->fmts[k].rate == r.rate && s->fmts[k].channels == r.channels) { *fmt = k; return AF_OK; }
    return fail(AF_ERR_INVALID, "record %zu: no admitted format is %u Hz x %u", i, r.rate, r.channels);
}
}  // namespace

extern "C" {

AF_API size_t af_session_stream_record_bytes(const af_session *s) { return s ? record_bytes(s) : 0; }

AF_API int af_session_export_streams(af_session *s, const uint32_t *streams, size_t n, void *records, int mem)
{
    if (!s || ((!streams || !records) && n)) return fail(AF_ERR_INVALID, "null argument");
    if (mem != AF_MEM_DEVICE && mem != AF_MEM_HOST) return fail(AF_ERR_INVALID, "bad memory kind %d", mem);
    for (size_t i = 0; i < n; ++i)
        if (streams[i] >= s->S) return fail(AF_ERR_INVALID, "stream index %u out of range (%zu streams)", streams[i], s->S);
    if (!n) return AF_OK;
    if (mem == AF_MEM_DEVICE && device_of_pointer(records) != s->device)
        return fail(AF_ERR_INVALID, "device records must live on the session's GPU %d", s->device);
    AF_SCOPE(s->device);
    cudaStream_t st = cur_ctx().stream;
    const size_t rb = record_bytes(s);
    int rc = reserve_transfer(s, n, mem == AF_MEM_DEVICE ? n : 0);
    if (rc) return rc;
    if (mem == AF_MEM_HOST) AF_CUDA(s->xfer.stage.grow(n * rb));
    std::vector<StreamRecord> hdr(n);
    RecordMove *mv = s->xfer.h_moves.get();
    for (size_t i = 0; i < n; ++i) {
        const uint32_t k = streams[i];
        const StreamState &c = s->diverged ? s->ss[k] : s->shared;
        StreamRecord &r = hdr[i];
        memset(&r, 0, sizeof(r));
        r.magic = REC_MAGIC; r.version = REC_VERSION; r.bytes = (uint32_t)rb;
        r.frame_len = s->frame_len; r.hop = s->hop;
        r.flags = framing_flags(s) | (c.restart ? REC_RESTART : 0u) | (s->wire && !c.restart ? REC_WIRE : 0u);
        r.rate = s->fmts[c.fmt].rate; r.channels = s->fmts[c.fmt].channels;
        r.vad = s->h_recs.get() ? s->vad_cfgs[k] : s->pipe->cfg.vad;
        mv[i] = RecordMove{k, c.in_drop, 0, c.y_drop, 0, 0};
        if (!c.restart) {                                        // a pending restart carries its format and configuration only
            memcpy(&r.last_index, &c.rec.last_index, sizeof(double));
            r.chunks = c.rec.chunks; r.n_out = c.rec.n_out;
            r.in_base = c.in_base; r.frames_emitted = c.frames_emitted;
            r.in_len = c.in_len; r.y_len = c.y_len;
            mv[i].in_len = c.in_len; mv[i].y_len = c.y_len;
        }
    }
    uint8_t *dst = mem == AF_MEM_HOST ? s->xfer.stage.get() : static_cast<uint8_t *>(records);
    AF_CUDA(cudaMemcpyAsync(s->xfer.d_moves.get(), mv, n * sizeof(RecordMove), cudaMemcpyHostToDevice, st));
    AF_CUDA(launch_session_pack(record_job(s, dst), (uint32_t)n, st));
    count_launch();
    const size_t H = sizeof(StreamRecord);
    if (mem == AF_MEM_HOST) {
        AF_CUDA(cudaMemcpy2DAsync(static_cast<uint8_t *>(records) + H, rb, dst + H, rb, rb - H, n, cudaMemcpyDeviceToHost, st));
    } else {
        memcpy(s->xfer.h_hdr.get(), hdr.data(), n * H);
        AF_CUDA(cudaMemcpy2DAsync(records, rb, s->xfer.h_hdr.get(), H, H, n, cudaMemcpyHostToDevice, st));
    }
    AF_CUDA(cudaStreamSynchronize(st));
    if (mem == AF_MEM_HOST)
        for (size_t i = 0; i < n; ++i) memcpy(static_cast<uint8_t *>(records) + i * rb, &hdr[i], H);
    return AF_OK;
}

AF_API int af_session_import_streams(af_session *s, const uint32_t *slots, const void *records, size_t n,
                                     const uint32_t *format, int mem)
{
    if (!s || ((!slots || !records) && n)) return fail(AF_ERR_INVALID, "null argument");
    if (mem != AF_MEM_DEVICE && mem != AF_MEM_HOST) return fail(AF_ERR_INVALID, "bad memory kind %d", mem);
    std::vector<uint8_t> seen(s->S, 0);
    for (size_t i = 0; i < n; ++i) {
        if (slots[i] >= s->S) return fail(AF_ERR_INVALID, "slot %u out of range (%zu streams)", slots[i], s->S);
        if (seen[slots[i]]++) return fail(AF_ERR_INVALID, "slot %u listed twice", slots[i]);
    }
    if (!n) return AF_OK;
    if (mem == AF_MEM_DEVICE && device_of_pointer(records) != s->device)
        return fail(AF_ERR_INVALID, "device records must live on the session's GPU %d", s->device);
    AF_SCOPE(s->device);
    cudaStream_t st = cur_ctx().stream;
    const size_t rb = record_bytes(s), H = sizeof(StreamRecord);
    int rc = reserve_transfer(s, n, mem == AF_MEM_DEVICE ? n : 0);
    if (rc) return rc;
    if (mem == AF_MEM_HOST) AF_CUDA(s->xfer.stage.grow(n * rb));
    // ---- the headers: read where they are (device records: one strided copy), every one checked before anything changes ----
    std::vector<StreamRecord> hdr(n);
    if (mem == AF_MEM_HOST) {
        for (size_t i = 0; i < n; ++i) memcpy(&hdr[i], static_cast<const uint8_t *>(records) + i * rb, H);
    } else {
        AF_CUDA(cudaMemcpy2DAsync(s->xfer.h_hdr.get(), H, records, rb, H, n, cudaMemcpyDeviceToHost, st));
        AF_CUDA(cudaStreamSynchronize(st));
        memcpy(hdr.data(), s->xfer.h_hdr.get(), n * H);
    }
    std::vector<uint32_t> fmt(n);
    for (size_t i = 0; i < n; ++i) {
        rc = check_record(s, hdr[i], i, format, &fmt[i]);
        if (rc) return rc;
    }
    // the configurations that travel: the tables exist once a record brings one other than the pipeline's
    if (s->pipe->cfg.vad_enable && !s->h_recs.get()) {
        const ScanRec base = scan_rec(s->pipe->vad_prm);
        std::vector<ScanRec> recs(n);
        std::vector<af_vad_config> cfgs(n);
        for (size_t i = 0; i < n; ++i) cfgs[i] = hdr[i].vad;
        make_scan_recs(cfgs.data(), n, recs.data());
        for (size_t i = 0; i < n && !s->h_recs.get(); ++i)
            if (!same_rec(recs[i], base)) {
                rc = alloc_vad_configs(s);
                if (rc) return rc;
            }
    }
    // ---- the device part: one launch scatters every record into the slots' current rows ----
    RecordMove *mv = s->xfer.h_moves.get();
    for (size_t i = 0; i < n; ++i)
        mv[i] = RecordMove{slots[i], 0, hdr[i].in_len, 0, hdr[i].y_len, (hdr[i].flags & REC_WIRE) ? 1u : 0u};
    s->wire_valid = s->levels_valid = false;                     // the last push's outputs no longer describe these slots
    const uint8_t *src = static_cast<const uint8_t *>(records);
    AF_CUDA(cudaMemcpyAsync(s->xfer.d_moves.get(), mv, n * sizeof(RecordMove), cudaMemcpyHostToDevice, st));
    if (mem == AF_MEM_HOST) {
        AF_CUDA(cudaMemcpy2DAsync(s->xfer.stage.get() + H, rb, src + H, rb, rb - H, n, cudaMemcpyHostToDevice, st));
        src = s->xfer.stage.get();
    }
    AF_CUDA(launch_session_unpack(record_job(s, const_cast<uint8_t *>(src)), (uint32_t)n, st));
    count_launch();
    if (s->wr.pre.frames) {                                      // a record carries no history: the import is an origin
        AF_CUDA(launch_session_preroll_clear(s->xfer.d_moves.get(), (uint32_t)n, s->wr.pre.d_n.get(), st));
        count_launch();
    }
    AF_CUDA(cudaStreamSynchronize(st));
    // ---- commit: the slots' bookkeeping, their configurations; lockstep again when every stream stands at one position ----
    if (!s->diverged) {
        s->ss.assign(s->S, s->shared);
        s->diverged = true;
    }
    for (size_t i = 0; i < n; ++i) {
        const StreamRecord &r = hdr[i];
        StreamState c = fresh_stream(s, fmt[i]);
        if (r.flags & REC_RESTART) {
            c.restart = true;                                    // the tick kernel clears history, detector and segment
        } else {
            memcpy(&c.rec.last_index, &r.last_index, sizeof(double));
            c.rec.chunks = r.chunks; c.rec.n_out = r.n_out;
            c.in_len = r.in_len; c.in_drop = 0;
            c.y_len = r.y_len; c.y_drop = 0;
            c.in_base = r.in_base; c.frames_emitted = r.frames_emitted;
        }
        s->ss[slots[i]] = c;
    }
    if (s->h_recs.get()) {
        std::vector<af_vad_config> cfgs(n);
        for (size_t i = 0; i < n; ++i) cfgs[i] = hdr[i].vad;
        put_vad_configs(s, slots, cfgs.data(), n);
    }
    bool aligned = true;
    for (size_t k = 0; k < s->S && aligned; ++k) aligned = same_position(s->ss[k], s->ss[0]);
    s->diverged = !aligned;
    if (aligned) s->shared = s->ss[0];
    return AF_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------
// level metering for the UI events (events/mod.rs:41,73-75 AudioLevel{level, peak}; modules/events/mod.rs:22,182-185
// VolumeLevel{level, is_speech}): by-products of a session tick
// ------------------------------------------------------------------------------------------
extern "C" {

AF_API int af_session_enable_levels(af_session *s, int enable)
{
    if (!s) return fail(AF_ERR_INVALID, "null session");
    AF_SCOPE(s->device);
    if (enable && !s->lv.d_peak.get()) {                 // all three buffers or none
        af_session::Levels lv;
        AF_CUDA(lv.d_peak.alloc(s->S));
        AF_CUDA(lv.h_peak.alloc(s->S));
        AF_CUDA(lv.h_vad.alloc(s->S));
        s->lv = std::move(lv);
    }
    s->levels = enable != 0;
    s->levels_valid = false;
    return AF_OK;
}

AF_API int af_session_levels(const af_session *s, float *level_db, float *peak, uint8_t *is_speech)
{
    if (!s) return fail(AF_ERR_INVALID, "null session");
    if (!s->levels_valid) return fail(AF_ERR_INVALID, "no tick has been pushed since af_session_enable_levels");
    const bool vad = s->pipe->cfg.vad_enable != 0;
    for (size_t k = 0; k < s->S; ++k) {
        if (peak) peak[k] = s->lv.h_peak.get()[k];
        // VoiceActivityDetector::energy_db (vad.rs:192-194) through energy_to_dbfs (vad.rs:171-176), host libm
        const VadState &v = s->lv.h_vad.get()[k];
        const float e = vad ? v.smoothed : 0.0f;
        if (level_db) level_db[k] = e <= 0.0f ? -INFINITY : 20.0f * log10f(e);
        if (is_speech) is_speech[k] = (vad && v.state == 1) ? 1 : 0;          // is_speaking, vad.rs:197-199
    }
    return AF_OK;
}

}  // extern "C"

namespace {
// The payload rows of w.cfg for a tick's payload and `pre` frames of pre-roll, into w: the session's rows stay as they
// are until the caller moves these in.  Ungated: the tick's new samples; gated: the hops of at most y_stride / hop + 2
// frames, plus the pre-roll's
int wire_rows(const af_session *s, uint32_t pre, af_session::Wire &w)
{
    const size_t S = s->S;
    w.cap = w.cfg.gate ? (s->y_stride / s->hop + 2 + pre) * s->hop : s->max_new_y;
    if (w.cfg.pcm16) {
        w.pcm16_stride = round_up(w.cap, 4);
        AF_CUDA(w.d_pcm16.alloc(S * w.pcm16_stride));
        if (w.cfg.mem == AF_MEM_HOST) AF_CUDA(w.h_pcm16.alloc(S * w.pcm16_stride));
    }
    if (w.cfg.base64) {
        w.b64_stride = round_up(af_pcm16_base64_len(w.cap), 4);
        AF_CUDA(w.d_b64.alloc(S * w.b64_stride));
        if (w.cfg.mem == AF_MEM_HOST) AF_CUDA(w.h_b64.alloc(S * w.b64_stride));
    }
    return AF_OK;
}

// The feature rows in `mem` for the frames of wire_rows(s, pre, .), into f
int feature_rows(const af_session *s, int mem, uint32_t pre, af_session::Wire::Features &f)
{
    const size_t S = s->S;
    f.mem = mem;
    f.stride = round_up((s->y_stride / s->hop + 2 + pre) * s->pipe->cfg.n_mels, 4);
    AF_CUDA(f.d_rows.alloc(S * f.stride));
    if (mem == AF_MEM_HOST) AF_CUDA(f.h_rows.alloc(S * f.stride));
    AF_CUDA(f.d_n.alloc(S));
    AF_CUDA(f.h_n.alloc(S));
    return AF_OK;
}

// The session takes w's payload rows and the pre-roll state `p` (once the device no longer writes the old ones); the
// last push's rows are gone with them
void take_wire_rows(af_session *s, af_session::Wire &w, af_session::Wire::Preroll &&p)
{
    af_session::Wire &wr = s->wr;
    wr.cap = w.cap;
    wr.d_pcm16 = std::move(w.d_pcm16); wr.h_pcm16 = std::move(w.h_pcm16); wr.pcm16_stride = w.pcm16_stride;
    wr.d_b64 = std::move(w.d_b64); wr.h_b64 = std::move(w.h_b64); wr.b64_stride = w.b64_stride;
    wr.pre = std::move(p);
    s->wire_valid = false;
    wr.feat.valid = false;
}
}  // namespace

extern "C" {

// ---- streaming wire output (websocket.rs:244-254 per tick): rows sized for the largest payload a tick can produce ----
AF_API int af_session_enable_wire(af_session *s, const af_wire_config *cfg)
{
    if (!s) return fail(AF_ERR_INVALID, "null session");
    AF_SCOPE(s->device);
    if (!cfg) {
        cudaDeviceSynchronize();                     // (a failed tick may still be writing the rows)
        wire_free(s);
        return AF_OK;
    }
    const af_pipeline_config &pc = s->pipe->cfg;
    if (cfg->gate > 1) return fail(AF_ERR_INVALID, "gate must be 0 or 1");
    if (cfg->gate && !pc.vad_enable) return fail(AF_ERR_INVALID, "the gated wire output needs the VAD (vad_enable)");
    if (cfg->gate && s->hop > s->frame_len)
        return fail(AF_ERR_INVALID, "the gated wire output needs vad_hop <= vad_frame_len (a completed frame's hop must have arrived)");
    if (!cfg->pcm16 && !cfg->base64) return fail(AF_ERR_INVALID, "the wire output needs pcm16 or base64");
    if (cfg->mem != AF_MEM_DEVICE && cfg->mem != AF_MEM_HOST) return fail(AF_ERR_INVALID, "bad memory kind %d", cfg->mem);
    cudaDeviceSynchronize();
    wire_free(s);
    const size_t S = s->S;
    af_session::Wire wr;                             // the session takes the rows once all of them are allocated
    wr.cfg = *cfg;
    int rc = wire_rows(s, 0, wr);
    if (rc) return rc;
    AF_CUDA(wr.d_ticks.alloc(S));
    AF_CUDA(wr.h_ticks.alloc(S));
    if (!s->d_wire_prev.get()) {                     // the carried segment state survives a re-enable, as the detector's does
        DevBuf<uint8_t> prev;
        AF_CUDA(prev.alloc(S));
        AF_CUDA(cudaMemset(prev.get(), 0, S));
        s->d_wire_prev = std::move(prev);
    }
    if (pc.vad_enable) AF_CUDA(s->d_states.grow(S * s->st_stride));   // the scan's states for the kernel
    s->wr = std::move(wr);
    s->wire = true;
    s->wire_valid = false;
    return AF_OK;
}

AF_API int af_session_wire(const af_session *s, const int16_t **pcm16, uint64_t *pcm16_stride, const char **base64,
                           uint64_t *base64_stride, af_wire_tick *ticks, uint64_t *first_frame)
{
    if (!s) return fail(AF_ERR_INVALID, "null session");
    if (!s->wire_valid) return fail(AF_ERR_INVALID, "no tick has been pushed since af_session_enable_wire");
    const af_session::Wire &wr = s->wr;
    const bool host = wr.cfg.mem == AF_MEM_HOST;
    if (pcm16) *pcm16 = host ? wr.h_pcm16.get() : wr.d_pcm16.get();
    if (pcm16_stride) *pcm16_stride = wr.pcm16_stride;
    if (base64) *base64 = host ? wr.h_b64.get() : wr.d_b64.get();
    if (base64_stride) *base64_stride = wr.b64_stride;
    if (ticks) memcpy(ticks, wr.h_ticks.get(), s->S * sizeof(af_wire_tick));
    if (first_frame) *first_frame = s->first_frames[0];
    return AF_OK;
}

// ---- wire features: the log-mel rows of the gated payload's frames, rows sized for the wire's bound of frames ----
AF_API int af_session_enable_wire_features(af_session *s, int enable, int mem)
{
    if (!s) return fail(AF_ERR_INVALID, "null session");
    AF_SCOPE(s->device);
    af_session::Wire rows;                           // the pre-roll goes back to 0: the payload rows without it
    rows.cfg = s->wr.cfg;
    if (!enable) {
        if (s->wr.pre.frames) {
            const int rc = wire_rows(s, 0, rows);
            if (rc) return rc;
        }
        cudaDeviceSynchronize();                     // (a failed tick may still be writing the rows)
        if (s->wr.pre.frames) take_wire_rows(s, rows, af_session::Wire::Preroll{});
        s->wr.feat = af_session::Wire::Features{};
        return AF_OK;
    }
    const af_pipeline_config &pc = s->pipe->cfg;
    if (!s->wire || !s->wr.cfg.gate) return fail(AF_ERR_INVALID, "wire features need the gated wire output (af_session_enable_wire, gate = 1)");
    if (!pc.n_mels || !pc.vad_enable) return fail(AF_ERR_INVALID, "wire features need log-mel features (n_mels) and the VAD");
    if (s->frame_len != WIN || s->hop != HOP)
        return fail(AF_ERR_INVALID, "wire features need the VAD on the STFT frames (vad_frame_len 0 or 400 / 160)");
    if (mem != AF_MEM_DEVICE && mem != AF_MEM_HOST) return fail(AF_ERR_INVALID, "bad memory kind %d", mem);
    af_session::Wire::Features f;                    // the session takes the rows once all of them are allocated
    int rc = feature_rows(s, mem, 0, f);             // the frames whose hops the gated wire rows hold
    if (rc) return rc;
    if (s->wr.pre.frames && (rc = wire_rows(s, 0, rows))) return rc;
    // (the tick's log-mel staging is grown by the tick that first needs it, before anything changes: what is allocated
    // here is exactly what disabling releases)
    cudaDeviceSynchronize();                        // (the rows replaced may still be written)
    if (s->wr.pre.frames) take_wire_rows(s, rows, af_session::Wire::Preroll{});
    s->wr.feat = std::move(f);
    return AF_OK;
}

// ---- wire pre-roll: every segment of the gated payload reaches back up to P frames (af_session_set_wire_preroll) ----
AF_API int af_session_set_wire_preroll(af_session *s, uint32_t frames)
{
    if (!s) return fail(AF_ERR_INVALID, "null session");
    if (!s->wire || !s->wr.cfg.gate) return fail(AF_ERR_INVALID, "the pre-roll needs the gated wire output (af_session_enable_wire, gate = 1)");
    if (frames > AF_WIRE_PREROLL_MAX) return fail(AF_ERR_INVALID, "pre-roll of %u frames (at most %u)", frames, AF_WIRE_PREROLL_MAX);
    AF_SCOPE(s->device);
    const size_t S = s->S;
    const af_session::Wire::Features &cur = s->wr.feat;
    // everything is allocated before anything changes: payload rows and feature rows that hold the pre-roll, the history
    af_session::Wire rows;
    rows.cfg = s->wr.cfg;
    int rc = wire_rows(s, frames, rows);
    if (rc) return rc;
    af_session::Wire::Features f;
    if (cur.d_rows.get() && (rc = feature_rows(s, cur.mem, frames, f))) return rc;
    af_session::Wire::Preroll p;
    p.frames = frames;
    if (frames) {
        AF_CUDA(p.d_pcm.alloc(S * frames * s->hop));
        if (cur.d_rows.get()) AF_CUDA(p.d_lm.alloc(S * frames * s->pipe->cfg.n_mels));
        AF_CUDA(p.d_n.alloc(S));
        AF_CUDA(p.d_pos.alloc(S));
        AF_CUDA(cudaMemset(p.d_n.get(), 0, S * sizeof(uint32_t)));   // every stream's origin is the next push
        AF_CUDA(cudaMemset(p.d_pos.get(), 0, S * sizeof(uint32_t)));
    }
    cudaDeviceSynchronize();                         // (the rows replaced may still be written)
    take_wire_rows(s, rows, std::move(p));
    if (cur.d_rows.get()) s->wr.feat = std::move(f);
    return AF_OK;
}

// ---- wire segments: the pieces of every segment in the gated payload, rows sized for the wire's bound of frames ----
AF_API int af_session_enable_wire_segments(af_session *s, int enable, int mem)
{
    if (!s) return fail(AF_ERR_INVALID, "null session");
    AF_SCOPE(s->device);
    if (!enable) {
        cudaDeviceSynchronize();                     // (a failed tick may still be writing the rows)
        s->wr.seg = af_session::Wire::Segments{};
        return AF_OK;
    }
    if (!s->wire || !s->wr.cfg.gate) return fail(AF_ERR_INVALID, "wire segments need the gated wire output (af_session_enable_wire, gate = 1)");
    if (mem != AF_MEM_DEVICE && mem != AF_MEM_HOST) return fail(AF_ERR_INVALID, "bad memory kind %d", mem);
    const size_t S = s->S;
    af_session::Wire::Segments g;                    // the session takes the rows once all of them are allocated
    g.mem = mem;
    // the frames of the payload rows without the pre-roll (T_max, as wire_rows), and at most ceil(T_max / 2) + 1 pieces:
    // the pre-roll adds frames to pieces, never pieces
    const uint64_t T_max = s->y_stride / s->hop + 2;
    g.stride = (T_max + 1) / 2 + 1;
    AF_CUDA(g.d_rows.alloc(S * g.stride));
    if (mem == AF_MEM_HOST) AF_CUDA(g.h_rows.alloc(S * g.stride));
    AF_CUDA(g.d_n.alloc(S));
    AF_CUDA(g.h_n.alloc(S));
    cudaDeviceSynchronize();                        // (the rows replaced may still be written)
    s->wr.seg = std::move(g);
    return AF_OK;
}

AF_API int af_session_wire_segments(const af_session *s, const af_wire_segment **rows, uint64_t *stride, uint32_t *n_segs)
{
    if (!s) return fail(AF_ERR_INVALID, "null session");
    const af_session::Wire::Segments &g = s->wr.seg;
    if (!s->wire_valid || !g.valid) return fail(AF_ERR_INVALID, "no tick has been pushed since af_session_enable_wire_segments");
    if (rows) *rows = g.mem == AF_MEM_HOST ? g.h_rows.get() : reinterpret_cast<const af_wire_segment *>(g.d_rows.get());
    if (stride) *stride = g.stride;
    if (n_segs) memcpy(n_segs, g.h_n.get(), s->S * sizeof(uint32_t));
    return AF_OK;
}

AF_API int af_session_wire_features(const af_session *s, const float **rows, uint64_t *stride, uint32_t *n_frames)
{
    if (!s) return fail(AF_ERR_INVALID, "null session");
    const af_session::Wire::Features &f = s->wr.feat;
    if (!s->wire_valid || !f.valid) return fail(AF_ERR_INVALID, "no tick has been pushed since af_session_enable_wire_features");
    if (rows) *rows = f.mem == AF_MEM_HOST ? f.h_rows.get() : f.d_rows.get();
    if (stride) *stride = f.stride;
    if (n_frames) memcpy(n_frames, f.h_n.get(), s->S * sizeof(uint32_t));
    return AF_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------
// capture hand-off: RingBuffer (capture.rs:84-161) in pinned host memory, feeding sessions
// ------------------------------------------------------------------------------------------
struct af_ring {
    float *buf = nullptr;
    PinnedBuf<float> pinned;                        // owns buf when it is pinned (else buf is malloc'ed)
    size_t capacity = 0;
    std::mutex mu;                                  // the reference locks its Vec for every call (capture.rs:103,124,159)
    std::atomic<size_t> write_pos{0}, read_pos{0};
};

namespace {
// (write_pos - read_pos + capacity) % capacity, as capture.rs:107-109,128,152
inline size_t ring_used(const af_ring *r)
{
    const size_t w = r->write_pos.load(std::memory_order_seq_cst), rd = r->read_pos.load(std::memory_order_seq_cst);
    return (w + r->capacity - rd) % r->capacity;
}
}  // namespace

extern "C" {

AF_API int af_ring_create(size_t capacity_samples, af_ring **out)
{
    if (!out) return fail(AF_ERR_INVALID, "null out pointer");
    // RingBuffer::new(0) builds, then every call divides by zero (capture.rs:108): refuse it here
    if (capacity_samples == 0) return fail(AF_ERR_INVALID, "ring capacity must be positive");
    af_ring *r = new af_ring;
    r->capacity = capacity_samples;
    // pinned when a device is bound (the session copies straight out of it), plain memory otherwise: the ring is a
    // host container, not a compute path
    if (cur_device() >= 0 && cur_ctx().ready && r->pinned.alloc(capacity_samples, cudaHostAllocPortable) == cudaSuccess) r->buf = r->pinned.get();
    else {
        cudaGetLastError();
        r->buf = static_cast<float *>(malloc(capacity_samples * sizeof(float)));
        if (!r->buf) { delete r; return fail(AF_ERR_INVALID, "out of memory for a ring of %zu samples", capacity_samples); }
    }
    memset(r->buf, 0, capacity_samples * sizeof(float));
    *out = r;
    return AF_OK;
}

AF_API void af_ring_destroy(af_ring *r)
{
    if (!r) return;
    if (!r->pinned.get()) free(r->buf);
    delete r;
}

AF_API size_t af_ring_capacity(const af_ring *r) { return r ? r->capacity : 0; }

// RingBuffer::write (capture.rs:101-121): keeps one slot free, drops what does not fit, returns the count written
AF_API size_t af_ring_write(af_ring *r, const float *data, size_t n)
{
    if (!r || (!data && n)) return 0;
    std::lock_guard<std::mutex> lk(r->mu);
    const size_t w = r->write_pos.load(std::memory_order_seq_cst);
    const size_t used = ring_used(r);
    const size_t avail = r->capacity - used;                 // saturating_sub: used < capacity always
    const size_t to_write = std::min(n, avail ? avail - 1 : 0);
    const size_t first = std::min(to_write, r->capacity - w);
    memcpy(r->buf + w, data, first * sizeof(float));
    memcpy(r->buf, data + first, (to_write - first) * sizeof(float));
    if (to_write) r->write_pos.store((w + to_write) % r->capacity, std::memory_order_seq_cst);
    return to_write;
}

// RingBuffer::read (capture.rs:123-147): AF_RING_EMPTY (not an error) is the reference's None; otherwise
// min(size, available) samples are copied out -- read(0) on a non-empty ring is Some(vec![])
AF_API int af_ring_read(af_ring *r, float *out, size_t size, size_t *n_read)
{
    if (!r || !n_read || (!out && size)) return fail(AF_ERR_INVALID, "null argument");
    std::lock_guard<std::mutex> lk(r->mu);
    const size_t rd = r->read_pos.load(std::memory_order_seq_cst);
    const size_t used = ring_used(r);
    *n_read = 0;
    if (used == 0) return AF_RING_EMPTY;
    const size_t to_read = std::min(size, used);
    const size_t first = std::min(to_read, r->capacity - rd);
    memcpy(out, r->buf + rd, first * sizeof(float));
    memcpy(out + first, r->buf, (to_read - first) * sizeof(float));
    r->read_pos.store((rd + to_read) % r->capacity, std::memory_order_seq_cst);
    *n_read = to_read;
    return AF_OK;
}

AF_API size_t af_ring_available(const af_ring *r) { return r ? ring_used(r) : 0; }   // capture.rs:149-154

AF_API void af_ring_clear(af_ring *r)                                                  // capture.rs:156-161
{
    if (!r) return;
    std::lock_guard<std::mutex> lk(r->mu);
    r->write_pos.store(0, std::memory_order_seq_cst);
    r->read_pos.store(0, std::memory_order_seq_cst);
    memset(r->buf, 0, r->capacity * sizeof(float));
}

// Reads counts[k] samples (none for 0) from each ring into row k of the session's pinned staging rows, *stride samples
// apart; a ring that yields fewer than it held a moment before fails the tick
static int read_rings(af_session *s, af_ring *const *rings, const uint32_t *counts, uint32_t max_count, uint64_t *stride)
{
    *stride = round_up(std::max<uint32_t>(max_count, 4), 4);
    AF_CUDA(s->ring_stage.grow(*stride * s->S));
    for (size_t k = 0; k < s->S; ++k) {
        if (!counts[k]) continue;
        size_t got = 0;
        const int rc = af_ring_read(rings[k], s->ring_stage.get() + k * *stride, counts[k], &got);
        if (rc != AF_OK || got != counts[k]) return fail(AF_ERR_INVALID, "ring %zu changed under the tick (another reader?)", k);
    }
    return AF_OK;
}

// One session tick fed by the capture rings: takes exactly n_samples from each of the session's n_streams rings
// (AudioCapturer::read_frame, capture.rs:310-319, for every stream at once) into the session's pinned staging rows
// and pushes them.  Nothing is consumed unless every ring holds n_samples.
AF_API int af_session_push_rings(af_session *s, af_ring *const *rings, uint32_t n_samples, const af_outputs *out,
                                 uint32_t *n_pcm, uint32_t *n_feat, uint32_t *n_vad)
{
    if (!s || !rings) return fail(AF_ERR_INVALID, "null argument");
    if (s->format != AF_FMT_F32) return fail(AF_ERR_INVALID, "capture rings hold f32 samples; the session was created for i16");
    for (size_t k = 0; k < s->S; ++k) {
        if (!rings[k]) return fail(AF_ERR_INVALID, "ring %zu is null", k);
        const size_t have = af_ring_available(rings[k]);
        if (have < n_samples) return fail(AF_ERR_INVALID, "ring %zu holds %zu samples, the tick needs %u", k, have, n_samples);
    }
    for (size_t k = 0; k < s->S; ++k) {                          // the push's count checks, before any ring is read
        const int rc = check_count(s, stream_fmt(s, k), n_samples, n_samples);
        if (rc) return rc;
    }
    s->counts.assign(s->S, n_samples);
    uint64_t stride = 0;
    const int rc = read_rings(s, rings, s->counts.data(), n_samples, &stride);
    if (rc) return rc;
    return af_session_push(s, s->ring_stage.get(), stride, n_samples, AF_MEM_HOST, out, n_pcm, n_feat, n_vad);
}

// AudioCapturer::read_frame(max) for every stream: each ring gives what it holds, up to max_samples, in whole frames
AF_API int af_session_push_rings_available(af_session *s, af_ring *const *rings, uint32_t max_samples, const uint8_t *end,
                                           const af_outputs *out, uint32_t *n_pcm, uint32_t *n_feat, uint32_t *n_vad)
{
    if (!s || !rings) return fail(AF_ERR_INVALID, "null argument");
    if (s->format != AF_FMT_F32) return fail(AF_ERR_INVALID, "capture rings hold f32 samples; the session was created for i16");
    if (max_samples > s->max_ring_samples)
        return fail(AF_ERR_CAPACITY, "max_samples %u exceeds the session's max_tick_samples", max_samples);
    s->counts.resize(s->S);
    for (size_t k = 0; k < s->S; ++k) {
        if (!rings[k]) return fail(AF_ERR_INVALID, "ring %zu is null", k);
        const af_session::Format &f = s->fmts[stream_fmt(s, k)];       // at most the stream's own bound, whole frames
        const size_t n = std::min<size_t>({max_samples, (size_t)f.channels * f.max_tick_frames, af_ring_available(rings[k])});
        s->counts[k] = (uint32_t)(n - n % f.channels);
    }
    uint64_t stride = 0;
    const int rc = read_rings(s, rings, s->counts.data(), max_samples, &stride);
    if (rc) return rc;
    return af_session_push_streams(s, s->ring_stage.get(), stride, s->counts.data(), end, AF_MEM_HOST, out, n_pcm, n_feat, n_vad);
}

}  // extern "C"
