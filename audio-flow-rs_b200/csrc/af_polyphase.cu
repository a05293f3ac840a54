// af_polyphase.cu -- anti-aliased polyphase resampling to 16 kHz for batches (af_batch_set_resampler with
// AF_RESAMPLE_POLYPHASE): the host design of the filter (scipy.signal.resample_poly's default) and the FIR kernel that
// writes a sub-batch's 16 kHz rows from its raw interleaved input.  The fused kernel then runs over those rows as
// 16 kHz mono f32 streams.
#include <cmath>
#include <numeric>

#include "af_device.cuh"
#include "af_launch.h"

namespace af {

// ------------------------------------------------------------------------------------------
// Filter design (host, f64): firwin(2L + 1, 1 / max(p, q), window=('kaiser', 5.0)), each tap cast to f32 and then
// scaled by (float)q in f32 -- the taps resample_poly(x, q, p) uses for f32 input.
// ------------------------------------------------------------------------------------------
namespace {

double bessel_i0(double x)           // power series; for x <= 5 the terms fall below 1e-17 of the sum within 30 steps
{
    const double h = 0.25 * x * x;
    double term = 1.0, sum = 1.0;
    for (int k = 1; k < 200 && term > 1e-18 * sum; ++k) {
        term *= h / ((double)k * (double)k);
        sum += term;
    }
    return sum;
}

}  // namespace

bool polyphase_ratio(uint32_t in_rate, uint32_t out_rate, uint32_t *p, uint32_t *q)
{
    if (in_rate == 0 || out_rate == 0) return false;
    const uint32_t g = std::gcd(in_rate, out_rate);
    *p = in_rate / g; *q = out_rate / g;
    return std::max(*p, *q) <= (uint32_t)POLY_MAX_RATIO;
}

void polyphase_filter(uint32_t p, uint32_t q, std::vector<float> *h)
{
    const uint32_t m = std::max(p, q);
    const long long L = 10ll * m, n = 2 * L + 1;
    const double fc = 1.0 / (double)m, beta = 5.0, i0b = bessel_i0(beta);
    std::vector<double> w(n);
    double sum = 0.0;
    for (long long i = 0; i < n; ++i) {
        const double t = (double)(i - L);                              // m - alpha of firwin
        const double x = fc * t;
        const double y = M_PI * (x == 0.0 ? 1.0e-20 : x);              // numpy.sinc
        const double r = t / (double)L;                                // kaiser: (n - alpha) / alpha
        w[i] = fc * (std::sin(y) / y) * (bessel_i0(beta * std::sqrt(1.0 - r * r)) / i0b);
        sum += w[i];
    }
    h->resize(n);
    const float scale = (float)q;
    for (long long i = 0; i < n; ++i) (*h)[i] = (float)(w[i] / sum) * scale;
}

// ------------------------------------------------------------------------------------------
// FIR kernel.  One CTA per tile of consecutive outputs of one stream: the CTA stages the downmixed input the tile
// needs (zero outside [0, n_in)) into shared memory, then y[n] = sum_k m[k] * h[n p + L - k q] over ascending k as a
// chain of fmaf from +0.
//   48 kHz (p = 3, q = 1): every output uses all 61 taps; they come from the kernel parameters (constant bank operands
//     of the FFMAs).  A thread computes FIR_HOT_R consecutive outputs from one pass over its window of staged samples,
//     so each sample is loaded from shared memory once for up to FIR_HOT_R FMAs; lanes sit 3 FIR_HOT_R = 21 samples
//     apart, an odd stride, so the loads are free of bank conflicts.  The outputs go back through shared memory and
//     leave as coalesced 16-byte stores.
//   other ratios: one output per thread; taps from shared memory when the table fits (FirStream::taps_smem), else
//     from global memory.
//   16 kHz (p = q = 1): the downmix is copied.
// ------------------------------------------------------------------------------------------
namespace {

template <bool SMEM_TAPS>
__device__ __forceinline__ void fir_generic(const FirStream &s, const float *__restrict__ xs, const float *__restrict__ h,
                                            uint32_t e0, uint32_t n_tile, float *__restrict__ y)
{
    const uint32_t p = s.p, q = s.q, two_l = 2 * s.L;
    for (uint32_t r = threadIdx.x; r < n_tile; r += FIR_THREADS) {
        const uint32_t d = (r * p + q - 1 - e0) / q;                   // first staged sample of output r
        uint32_t j = two_l + r * p - e0 - d * q;                        // its tap: the largest index <= 2L of the phase
        const float *x = xs + d;
        float acc = 0.0f;
        for (;;) {
            acc = fmaf(*x++, SMEM_TAPS ? h[j] : __ldg(h + j), acc);
            if (j < q) break;
            j -= q;
        }
        y[r] = acc;
    }
}

}  // namespace

__global__ void __launch_bounds__(FIR_THREADS) af_polyphase_fir_kernel(const __grid_constant__ FirJob J)
{
    extern __shared__ float4 fir_smem[];
    float *sm = reinterpret_cast<float *>(fir_smem);
    const uint2 tile = J.tiles[blockIdx.x];
    const FirStream &s = J.streams[tile.x];
    const uint64_t n0 = (uint64_t)tile.y * s.tile_out;
    const uint32_t n_tile = min(s.tile_out, s.n_out - (uint32_t)n0);
    const bool copy = s.p == 1 && s.q == 1;
    const bool hot = s.p == 3 && s.q == 1;

    // staged input m[base .. base + span): base is the first input of output n0, e0 = base q - (n0 p - L) in [0, q)
    long long base = (long long)n0;
    uint32_t e0 = 0, span = n_tile;
    if (!copy) {
        const long long t = (long long)n0 * s.p - s.L;
        base = t >= 0 ? (t + s.q - 1) / s.q : -(-t / (long long)s.q);
        e0 = (uint32_t)(base * s.q - t);
        span = (uint32_t)(((long long)(n0 + n_tile - 1) * s.p + s.L) / s.q - base + 1);
    }
    const long long k_a = base & ~3ll;                                  // 16-byte aligned start of the stage
    const uint32_t o = (uint32_t)(base - k_a);
    const uint32_t n4 = (o + span + 3) / 4;
    if (s.channels == 1 && s.format == FMT_F32) {
        const float *x = static_cast<const float *>(s.data);
        for (uint32_t i = threadIdx.x; i < n4; i += FIR_THREADS) {
            const long long k = k_a + 4ll * i;
            float4 v;
            if (k >= 0 && k + 4 <= (long long)s.n_in) v = __ldg(reinterpret_cast<const float4 *>(x + k));
            else {
                v.x = k >= 0 && k < s.n_in ? __ldg(x + k) : 0.0f;
                v.y = k + 1 >= 0 && k + 1 < s.n_in ? __ldg(x + k + 1) : 0.0f;
                v.z = k + 2 >= 0 && k + 2 < s.n_in ? __ldg(x + k + 2) : 0.0f;
                v.w = k + 3 >= 0 && k + 3 < s.n_in ? __ldg(x + k + 3) : 0.0f;
            }
            fir_smem[i] = v;
        }
    } else {
        for (uint32_t i = threadIdx.x; i < 4 * n4; i += FIR_THREADS) {
            const long long k = k_a + i;
            sm[i] = k >= 0 && k < s.n_in ? load_mono(s.data, s.n_samples, s.n_in, s.channels, s.format, (int)k) : 0.0f;
        }
    }
    float *aux = sm + 4 * n4;                                           // taps (other ratios) or outputs (48 kHz)
    if (!copy && !hot && s.taps_smem)
        for (uint32_t i = threadIdx.x; i <= 2 * s.L; i += FIR_THREADS) aux[i] = __ldg(s.h + i);
    __syncthreads();

    const float *xs = sm + o;
    float *y = s.y + n0;
    if (copy) {
        for (uint32_t r = threadIdx.x; r < n_tile; r += FIR_THREADS) y[r] = xs[r];
    } else if (hot) {
        const float *w = xs + 3 * FIR_HOT_R * threadIdx.x;
        float acc[FIR_HOT_R];
#pragma unroll
        for (int r = 0; r < FIR_HOT_R; ++r) acc[r] = 0.0f;
#pragma unroll
        for (int i = 0; i < 3 * (FIR_HOT_R - 1) + FIR_HOT_TAPS; ++i) {
            const float v = w[i];
#pragma unroll
            for (int r = 0; r < FIR_HOT_R; ++r) {
                const int j = FIR_HOT_TAPS - 1 - i + 3 * r;             // output r's tap for sample i of the window
                if (j >= 0 && j < FIR_HOT_TAPS) acc[r] = fmaf(v, J.h3[j], acc[r]);
            }
        }
#pragma unroll
        for (int r = 0; r < FIR_HOT_R; ++r) aux[FIR_HOT_R * threadIdx.x + r] = acc[r];
        __syncthreads();
        // rows are 16-byte aligned and n0 is a multiple of 4
        const uint32_t n_vec = n_tile / 4;
        for (uint32_t i = threadIdx.x; i < n_vec; i += FIR_THREADS)
            reinterpret_cast<float4 *>(y)[i] = reinterpret_cast<const float4 *>(aux)[i];
        for (uint32_t r = 4 * n_vec + threadIdx.x; r < n_tile; r += FIR_THREADS) y[r] = aux[r];
    } else if (s.taps_smem) {
        fir_generic<true>(s, xs, aux, e0, n_tile, y);
    } else {
        fir_generic<false>(s, xs, s.h, e0, n_tile, y);
    }
}

uint32_t fir_tile_outputs(uint32_t p, uint32_t q)
{
    if (p == 3 && q == 1) return FIR_HOT_TILE;
    if (p == 1 && q == 1) return FIR_TILE_MAX;
    // the stage of a tile of T outputs holds at most ((T - 1) p + 2L) / q + 2 samples, plus up to 6 of alignment
    const uint64_t two_l = 20ull * std::max(p, q);
    uint64_t T = FIR_TILE_MAX;
    while (T > 4 && ((T - 1) * p + two_l) / q + 8 > (uint64_t)FIR_STAGE_MAX) T -= 4;
    return (uint32_t)T;
}

size_t fir_smem_floats(uint32_t p, uint32_t q, bool taps_smem)
{
    const uint64_t T = fir_tile_outputs(p, q);
    const uint64_t stage = p == 1 && q == 1 ? T + 8 : ((T - 1) * p + 20ull * std::max(p, q)) / q + 8;
    const uint64_t aux = p == 3 && q == 1 ? FIR_HOT_TILE : (taps_smem ? 20ull * std::max(p, q) + 1 : 0);
    return (size_t)((stage + 3) / 4 * 4 + aux);
}

cudaError_t launch_polyphase_fir(const FirJob &job, cudaStream_t st)
{
    if (job.n_tiles == 0) return cudaSuccess;
    const size_t bytes = job.smem_floats * sizeof(float);
    if (bytes > 48 * 1024) {
        const cudaError_t e = cudaFuncSetAttribute(af_polyphase_fir_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
        if (e != cudaSuccess) return e;
    }
    af_polyphase_fir_kernel<<<job.n_tiles, FIR_THREADS, bytes, st>>>(job);
    return cudaGetLastError();
}

}  // namespace af
