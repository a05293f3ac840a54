// af_internal.h -- what the translation units of the host runtime share (af_runtime.cu, af_multi.cu): the
// per-device library contexts, error plumbing and the internal form of a batch run.  Not part of the C ABI.
#pragma once
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <utility>
#include <vector>

#include "../../include/audioflow_gpu.h"
#include "af_device.cuh"
#include "af_launch.h"
#include "af_plan.h"

namespace afrt {

using namespace af;

constexpr int MAX_DEV = AF_MAX_GPUS;

int fail(int code, const char *fmt, ...);

#define AF_CUDA(expr)                                                                              \
    do {                                                                                           \
        cudaError_t _e = (expr);                                                                   \
        if (_e != cudaSuccess) return ::afrt::fail(AF_ERR_CUDA, "CUDA error %s at %s:%d: %s", #expr, __FILE__, __LINE__, \
                                                   cudaGetErrorString(_e));                        \
    } while (0)

// Every device and pinned allocation of the library is owned by a Buf: move-only, freed when the owner is reset,
// reassigned or destroyed.  g_live_allocs counts the live allocations of each kind (af_debug_live_allocations): the
// one leak check that works on a GPU other processes share.
enum class Mem { Device, Pinned };
inline std::atomic<uint64_t> g_live_allocs[2]{};

template <class T, Mem K>
class Buf {
  public:
    Buf() = default;
    Buf(Buf &&o) noexcept : p_(o.p_), n_(o.n_) { o.p_ = nullptr; o.n_ = 0; }
    Buf &operator=(Buf &&o) noexcept
    {
        if (this != &o) {
            reset();
            std::swap(p_, o.p_);
            std::swap(n_, o.n_);
        }
        return *this;
    }
    ~Buf() { reset(); }

    T *get() const { return p_; }
    size_t size() const { return n_; }             // elements

    // n elements in place of what the owner held (host_flags: cudaHostAlloc's, pinned only); empty on failure
    cudaError_t alloc(size_t n, unsigned host_flags = cudaHostAllocDefault)
    {
        reset();
        void *p = nullptr;
        const cudaError_t e = K == Mem::Device ? cudaMalloc(&p, n * sizeof(T)) : cudaHostAlloc(&p, n * sizeof(T), host_flags);
        if (e != cudaSuccess) return e;
        p_ = static_cast<T *>(p);
        n_ = n;
        if (p_) g_live_allocs[(int)K].fetch_add(1, std::memory_order_relaxed);
        return cudaSuccess;
    }
    // at least n elements: reallocates only when n exceeds the size, and does not keep the contents
    cudaError_t grow(size_t n) { return n <= n_ ? cudaSuccess : alloc(n); }

    cudaError_t reset()
    {
        if (!p_) return cudaSuccess;
        const cudaError_t e = K == Mem::Device ? cudaFree(p_) : cudaFreeHost(p_);
        if (e == cudaSuccess) g_live_allocs[(int)K].fetch_sub(1, std::memory_order_relaxed);
        p_ = nullptr;
        n_ = 0;
        return e;
    }

    // af_host_alloc hands an allocation to the caller and af_host_free takes it back: it stays counted meanwhile
    T *release()
    {
        T *p = p_;
        p_ = nullptr;
        n_ = 0;
        return p;
    }
    static Buf adopt(T *p)
    {
        Buf b;
        b.p_ = p;
        return b;
    }

  private:
    T *p_ = nullptr;
    size_t n_ = 0;
};

template <class T> using DevBuf = Buf<T, Mem::Device>;
template <class T> using PinnedBuf = Buf<T, Mem::Pinned>;

struct FracTable {                    // device copy of the f32 fractional offsets of one rate pair
    DevBuf<float> d;
    size_t n = 0;
};

struct RatePlan {                     // batch-path plan of one (in, out) pair, grown on demand
    RsRecurrence rec;                 // state after cum.size() - 1 chunks
    std::vector<uint64_t> cum{0};     // cum[c] = outputs after c chunks (table mode)
    std::vector<float> frac;          // host copy (table mode)
    std::shared_ptr<FracTable> dev;   // device copy covering frac.size() entries
};

// One context per GPU the process uses.  A thread works on ONE device at a time: the one it selected with af_init /
// af_init_multi, or the one the handle it passes was created on (DevScope).  The contexts live until the process ends
// and are never destroyed: af_shutdown releases what they hold.
struct Context {
    bool ready = false;
    int device = -1;
    int sm_count = 148;
    cudaStream_t stream = nullptr;    // the stream the library enqueues on: its own (non-blocking) one, or the caller's (af_set_stream)
    cudaStream_t own = nullptr;
    cudaStream_t side = nullptr;      // second stream: the result gather runs here, off the compute stream
    DevBuf<FftTables> d_fft;
    std::mutex mu;                    // guards the scratch buffers and the plan cache
    DevBuf<uint8_t> scratch_in, scratch_out, scratch_aux, scratch_jobs;
    std::map<uint64_t, RatePlan> plans;
};

Context &cur_ctx();                   // context of the device this thread works on (valid after require_ctx / DevScope)
int cur_device();                     // ... and its index (-1: none yet)
int require_ctx();                    // selects (initialising on first use) the thread's device; AF_OK or an error
int init_device(int device);          // initialises `device` (idempotent) WITHOUT selecting it
Context *device_ctx(int device);      // nullptr when not initialised

// Makes `dev` the device of the calling thread (CUDA's and the library's) for the lifetime of the object and restores
// both afterwards: entry points that take a handle run on the device the handle was created on.
struct DevScope {
    int prev_lib, prev_cuda, dev;
    int rc;
    explicit DevScope(int dev_);
    ~DevScope();
};

#define AF_SCOPE(dev_)                      \
    ::afrt::DevScope scope_((dev_));        \
    if (scope_.rc != AF_OK) return scope_.rc

void count_launch(uint64_t n = 1);
const std::string &kernel_variant();

// device a device pointer lives on (-1: not a device pointer / unknown)
int device_of_pointer(const void *p);

// af_batch_run on an explicit stream with the VAD states written to `vad` (may differ from o->vad: the sharded
// batches point it into the gather buffer).  Never synchronises.
int batch_run_on(af_batch *b, const af_outputs *o, uint8_t *vad, uint64_t vad_stride, cudaStream_t st);
int batch_device(const af_batch *b);
int batch_check_outputs(const af_batch *b, const af_outputs *o);
const af_pipeline_config &pipeline_cfg(const af_pipeline *p);
int plan_stream_counts(const af_pipeline_config &cfg, const af_stream_desc &d, uint32_t *n_out, uint32_t *n_frames, uint32_t *n_vad);
uint64_t batch_max_vad(const af_batch *b);

// the communicator side (af_multi.cu)
void comm_shutdown_all();

}  // namespace afrt
