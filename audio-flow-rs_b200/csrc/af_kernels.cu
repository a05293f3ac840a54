// af_kernels.cu -- the small kernels around the fused path: compat objects (to_mono, chunked
// resampling, single-detector VAD), generic frame energies, the sequential VAD scan, PCM16
// encode and VAD segmentation.
#include <cstdio>
#include "af_device.cuh"
#include "af_launch.h"

#include <cmath>

namespace af {

// ---- AudioFrame::to_mono (capture.rs:30-42) on a device buffer ----
__global__ void af_to_mono_kernel(const float *__restrict__ in, uint64_t n_samples, uint32_t channels,
                                  float *__restrict__ out, uint64_t n_frames)
{
    for (uint64_t f = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; f < n_frames;
         f += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t base = f * channels;
        uint32_t m = channels;
        if (base + m > n_samples) m = (uint32_t)(n_samples - base);
        float sum = 0.0f;
        for (uint32_t c = 0; c < m; ++c) sum = __fadd_rn(sum, in[base + c]);
        out[f] = channels == 1 ? in[f] : __fdiv_rn(sum, (float)channels);
    }
}

cudaError_t launch_to_mono(const float *in, uint64_t n_samples, uint32_t channels, float *out, uint64_t n_frames,
                           cudaStream_t st)
{
    if (n_frames == 0) return cudaSuccess;
    const int blocks = (int)std::min<uint64_t>((n_frames + 255) / 256, 148 * 8);
    af_to_mono_kernel<<<blocks, 256, 0, st>>>(in, n_samples, channels, out, n_frames);
    return cudaGetLastError();
}

// ---- generic chunk-exact resampling of mono device signals (AudioResampler / BatchResampler /
//      sessions): one thread per output sample, blockIdx.y = job ----
__global__ void af_resample_jobs_kernel(const ResampleJob *__restrict__ jobs)
{
    const ResampleJob J = jobs[blockIdx.y];
    const unsigned long long count = J.n_end - J.n_begin;
    for (unsigned long long o = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; o < count;
         o += (unsigned long long)gridDim.x * blockDim.x) {
        const unsigned long long n = J.n_begin + o;
        if (J.mode == RS_PASSTHROUGH) {
            const long long idx = (long long)n;
            J.out[o] = (idx < J.data_base || idx >= J.n_valid_end) ? 0.0f : J.data[idx - J.data_base];
            continue;
        }
        long long k; uint32_t rem;
        resample_pos(n, J.p, J.q, &k, &rem);
        float frac;
        if (J.mode == RS_TABLE) {
            frac = J.frac[n];
            if (rem == 0 && frac >= 0.5f) k -= 1;
        } else {
            frac = (float)rem * (1.0f / (float)J.q);
        }
        float y[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            const long long idx = k - 1 + t;
            y[t] = (idx < J.data_base || idx >= J.n_valid_end) ? 0.0f : J.data[idx - J.data_base];
        }
        J.out[o] = interp_cubic(frac, y[0], y[1], y[2], y[3]);
    }
}

cudaError_t launch_resample_jobs(const ResampleJob *jobs_dev, uint32_t n_jobs, uint32_t max_outputs, cudaStream_t st)
{
    if (n_jobs == 0 || max_outputs == 0) return cudaSuccess;
    dim3 grid(std::min<uint32_t>((max_outputs + 255) / 256, 1024), n_jobs);
    af_resample_jobs_kernel<<<grid, 256, 0, st>>>(jobs_dev);
    return cudaGetLastError();
}

// ---- calculate_energy (vad.rs:157-168) for arbitrary (frame_len, hop): one thread per frame ----
__global__ void af_frame_energy_kernel(const EnergyJob J)
{
    const uint32_t s = blockIdx.y;
    const uint32_t T = J.n_frames ? J.n_frames[s] : J.n_frames_all;
    const float *y = J.y + (uint64_t)s * J.y_stride;
    float *e = J.energy + (uint64_t)s * J.energy_stride;
    for (uint32_t f = blockIdx.x * blockDim.x + threadIdx.x; f < T; f += gridDim.x * blockDim.x) {
        const float *x = y + (uint64_t)f * J.hop;
        float sum = 0.0f;
        for (uint32_t i = 0; i < J.frame_len; ++i) {
            const float v = x[i];
            sum = __fadd_rn(sum, __fmul_rn(v, v));
        }
        e[f] = J.frame_len ? __fdiv_rn(sum, (float)J.frame_len) : 0.0f;
    }
}

cudaError_t launch_frame_energy(const EnergyJob &job, cudaStream_t st)
{
    if (job.n_streams == 0) return cudaSuccess;
    uint32_t maxT = job.n_frames_all ? job.n_frames_all : 1;
    dim3 grid(std::min<uint32_t>((maxT + 127) / 128, 2048), job.n_streams);
    af_frame_energy_kernel<<<grid, 128, 0, st>>>(job);
    return cudaGetLastError();
}

// ---- detect() EMA + threshold + state machine (vad.rs:101-153): strictly sequential per stream ----
// One thread per stream; latency bound.  Per 32 frames: (1) the EMA chain (fmul, fadd per frame, the only
// floating-point recurrence) produces a word of is_speech bits, (2) the state machine consumes the word
// RUN BY RUN (ffs on the bit word) instead of frame by frame: a run of equal decisions changes the state at
// most once (Silence->Speech on the first 1, Speech->Ending/Silence on the zero that reaches the timeout).
struct VadMachine {        // 32-bit working copy of (state, silence_frames, speech_frames); see the overflow guard below
    uint32_t st, sil, spk;
};

__device__ __forceinline__ void vad_emit(uint8_t *out, uint32_t f, uint32_t count, uint32_t v)
{
    if (!out) return;
    for (uint32_t i = 0; i < count; ++i) out[f + i] = (uint8_t)v;     // independent byte stores
}

// consumes n (<= 32) decisions, bit j of `bits` = frame f0 + j; exact vad.rs:121-153 semantics
__device__ __forceinline__ void vad_machine_word(VadMachine &m, uint32_t bits, uint32_t n, uint32_t f0, uint8_t *out,
                                                 uint32_t timeout, uint32_t min_speech)
{
    uint32_t j = 0;
    while (j < n) {
        const uint32_t rem = bits >> j;                   // bit 0 = decision of frame j (bits above n are zero)
        if (m.st == 0u) {                                 // Silence: zeros keep it; the first 1 enters Speech
            if (rem == 0u) { vad_emit(out, f0 + j, n - j, 0u); j = n; break; }
            const uint32_t z = (uint32_t)__ffs((int)rem) - 1u;
            vad_emit(out, f0 + j, z, 0u);
            m.st = 1u; m.spk = 1u; m.sil = 0u;
            vad_emit(out, f0 + j + z, 1u, 1u);
            j += z + 1u;
        } else if (m.st == 1u) {
            if (rem & 1u) {                               // run of speech frames
                uint32_t r = (uint32_t)__ffs((int)~rem) - 1u;        // ~rem != 0 or ffs gives 0 -> r = 0xffffffff
                if (~rem == 0u) r = 32u;
                r = min(r, n - j);
                m.spk += r; m.sil = 0u;
                vad_emit(out, f0 + j, r, 1u);
                j += r;
            } else {                                      // run of non-speech frames
                uint32_t r = rem ? (uint32_t)__ffs((int)rem) - 1u : 32u;
                r = min(r, n - j);
                const uint32_t need = timeout > m.sil ? timeout - m.sil : 1u;   // zeros until silence_frames >= timeout
                if (r < need) {
                    m.sil += r;
                    vad_emit(out, f0 + j, r, 1u);
                    j += r;
                } else {
                    vad_emit(out, f0 + j, need - 1u, 1u);
                    m.sil += need;
                    m.st = m.spk >= min_speech ? 2u : 0u;
                    m.spk = 0u;
                    vad_emit(out, f0 + j + need - 1u, 1u, m.st);
                    j += need;
                }
            }
        } else {                                          // Ending: one frame, whatever it is
            m.st = 0u; m.sil = 0u;
            vad_emit(out, f0 + j, 1u, 0u);
            j += 1u;
        }
    }
}

// flagged_only: the launch after the parallel kernel of a job with per-stream records takes only the streams flagged seq
__global__ void af_vad_scan_kernel(const ScanJob J, uint32_t flagged_only)
{
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= J.n_streams) return;
    if (flagged_only && !J.recs[s].seq) return;
    const uint32_t T = J.n_frames ? J.n_frames[s] : J.n_frames_all;
    const float *e = J.energy + (uint64_t)s * J.energy_stride;
    uint8_t *out = J.states ? J.states + (uint64_t)s * J.states_stride : nullptr;
    VadState v;
    if (J.state_io) v = J.state_io[s];
    else { v.smoothed = 0.0f; v.state = 0; v.silence_frames = 0; v.speech_frames = 0; }
    const VadParams prm = J.recs ? J.recs[s].prm : J.prm;
    // the fast path keeps the counters in 32 bits; fall back to the plain 64-bit step when they could overflow
    const bool small = v.silence_frames < 0x40000000ull && v.speech_frames < 0x40000000ull && T < 0x40000000u &&
                       prm.silence_timeout < 0x40000000ull && prm.min_speech < 0x80000000ull;
    if (!small) {
        for (uint32_t f = 0; f < T; ++f) {
            const int stv = vad_step(v, prm, e[f]);
            if (out) out[f] = (uint8_t)stv;
        }
        if (J.state_io) J.state_io[s] = v;
        if (J.final_out) J.final_out[s] = v;
        return;
    }
    const float alpha = prm.alpha, beta = __fsub_rn(1.0f, prm.alpha), e_min = prm.e_min;
    const bool use_smoothed = alpha > 0.0f;
    float sm = v.smoothed;
    VadMachine m{(uint32_t)v.state, (uint32_t)v.silence_frames, (uint32_t)v.speech_frames};
    const uint32_t timeout = (uint32_t)prm.silence_timeout, minsp = (uint32_t)prm.min_speech;
    uint32_t f = 0;
    const bool vec_in = ((reinterpret_cast<uintptr_t>(e) & 15) == 0);
    if (vec_in && T >= 32) {
        const float4 *e4 = reinterpret_cast<const float4 *>(e);
        const uint32_t n_words = T / 32;
        float4 cur[8], nxt[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) cur[j] = e4[j];
        for (uint32_t w = 0; w < n_words; ++w) {
            if (w + 1 < n_words) {
#pragma unroll
                for (int j = 0; j < 8; ++j) nxt[j] = e4[(w + 1) * 8 + j];       // prefetch the next 32 energies
            }
            uint32_t bits = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) {                 // EMA chain (vad.rs:101-118)
                const float ev[4] = {cur[j].x, cur[j].y, cur[j].z, cur[j].w};
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    sm = __fadd_rn(__fmul_rn(alpha, ev[c]), __fmul_rn(beta, sm));
                    bits |= ((use_smoothed ? sm : ev[c]) >= e_min ? 1u : 0u) << (4 * j + c);
                }
            }
            vad_machine_word(m, bits, 32u, w * 32u, out, timeout, minsp);
#pragma unroll
            for (int j = 0; j < 8; ++j) cur[j] = nxt[j];
        }
        f = n_words * 32;
    }
    while (f < T) {                                       // tail (and unaligned rows): up to 32 frames at a time
        const uint32_t n = min(32u, T - f);
        uint32_t bits = 0;
        for (uint32_t j = 0; j < n; ++j) {
            const float ev = e[f + j];
            sm = __fadd_rn(__fmul_rn(alpha, ev), __fmul_rn(beta, sm));
            bits |= ((use_smoothed ? sm : ev) >= e_min ? 1u : 0u) << j;
        }
        vad_machine_word(m, bits, n, f, out, timeout, minsp);
        f += n;
    }
    v.smoothed = sm; v.state = (int)m.st; v.silence_frames = m.sil; v.speech_frames = m.spk;
    if (J.state_io) J.state_io[s] = v;
    if (J.final_out) J.final_out[s] = v;
}

// ---- the same scan, parallel inside a stream: one CTA per stream -------------------------------------------
// The EMA is the only floating-point recurrence.  It is cut into chunks of SCAN_CHUNK frames; every chunk but the
// first of a block starts `warm` frames early from 0 and must arrive at its first frame with EXACTLY (bit for bit)
// the value the previous chunk ended with -- the influence of the unknown start decays as (1 - alpha)^warm, far
// below one ulp for the warm-up lengths chosen by the host.  Each boundary is verified; a block with a mismatch
// is recomputed sequentially by one thread, so the result never depends on the speculation.  The decisions
// (one bit per frame) then drive the state machine: one thread walks the bit words run by run and records
// the machine state at every word boundary, after which every thread expands its own words into state bytes.
// The energies of a block (and of the warm-up before it) are first copied to shared memory with coalesced loads: the
// chains then read them at shared-memory latency instead of paying a dependent global load per frame (a one-hour
// stream, 360 000 frames through one CTA, went from 2.48 ms to 0.3 ms).
constexpr uint32_t SCAN_CHUNK = 64;                  // frames per EMA chunk (2 bit words): one chunk per thread and block
constexpr uint32_t SCAN_BLOCK = 8192;                // frames per block of a long stream (128 chunks, 256 words)
constexpr uint32_t SCAN_THREADS = 128;
constexpr uint32_t SCAN_WARM_MAX = 512;              // longest warm-up the host selects (scan_warmup)
// The staged energies are read by one thread per chunk, i.e. SCAN_CHUNK (= two banks' worth of) floats apart: without
// padding every lane of a warp hits the same bank (measured: 112 cycles per EMA step).  One pad word per SCAN_CHUNK floats
// puts the lanes on consecutive banks.
__host__ __device__ constexpr uint32_t epad(uint32_t i) { return i + i / SCAN_CHUNK; }
constexpr uint32_t SCAN_E_FLOATS = epad(SCAN_WARM_MAX + SCAN_BLOCK) + 1;
// EB(x) = e[b0 + x] for x in [-lead, n): the block's energies (and the warm-up in front of it) staged in s_e
#define EB(x) s_e[epad((uint32_t)((int)lead + (int)(x)))]

struct EmitMask {          // collects the states of one word as two bit masks (Speech, Ending)
    uint32_t speech = 0, ending = 0;
    __device__ __forceinline__ void run(uint32_t j, uint32_t count, uint32_t v)
    {
        if (count == 0 || v == 0u) return;
        const uint32_t m = (count >= 32u ? 0xffffffffu : ((1u << count) - 1u)) << j;
        if (v == 1u) speech |= m; else ending |= m;
    }
};
struct EmitNone {
    __device__ __forceinline__ void run(uint32_t, uint32_t, uint32_t) {}
};

// vad_machine_word with a pluggable sink; j counts from the start of the word
template <class Emit>
__device__ __forceinline__ void vad_machine_word_t(VadMachine &m, uint32_t bits, uint32_t n, Emit &em, uint32_t timeout,
                                                   uint32_t min_speech)
{
    uint32_t j = 0;
    while (j < n) {
        const uint32_t rem = bits >> j;
        if (m.st == 0u) {
            if (rem == 0u) { em.run(j, n - j, 0u); j = n; break; }
            const uint32_t z = (uint32_t)__ffs((int)rem) - 1u;
            em.run(j, z, 0u);
            m.st = 1u; m.spk = 1u; m.sil = 0u;
            em.run(j + z, 1u, 1u);
            j += z + 1u;
        } else if (m.st == 1u) {
            if (rem & 1u) {
                uint32_t r = (~rem == 0u) ? 32u : (uint32_t)__ffs((int)~rem) - 1u;
                r = min(r, n - j);
                m.spk += r; m.sil = 0u;
                em.run(j, r, 1u);
                j += r;
            } else {
                uint32_t r = rem ? (uint32_t)__ffs((int)rem) - 1u : 32u;
                r = min(r, n - j);
                const uint32_t need = timeout > m.sil ? timeout - m.sil : 1u;
                if (r < need) {
                    m.sil += r;
                    em.run(j, r, 1u);
                    j += r;
                } else {
                    em.run(j, need - 1u, 1u);
                    m.sil += need;
                    m.st = m.spk >= min_speech ? 2u : 0u;
                    m.spk = 0u;
                    em.run(j + need - 1u, 1u, m.st);
                    j += need;
                }
            }
        } else {
            m.st = 0u; m.sil = 0u;
            em.run(j, 1u, 0u);
            j += 1u;
        }
    }
}

// EMA over frames [f0, f1) of the staged energies (x = f - b0), strictly sequential (vad.rs:101-106); the loads of four
// steps are issued ahead of their dependent multiply-add chain.  `ema_bits` also collects up to 32 decision bits.
#define AF_EMA_STEP(sm, ev) __fadd_rn(__fmul_rn(alpha, (ev)), __fmul_rn(beta, (sm)))
__device__ __forceinline__ float ema_run(const float *s_e, uint32_t lead, int x0, int x1, float sm, float alpha, float beta)
{
    int x = x0;
    for (; x + 4 <= x1; x += 4) {
        const float e0 = EB(x), e1 = EB(x + 1), e2 = EB(x + 2), e3 = EB(x + 3);
        sm = AF_EMA_STEP(sm, e0); sm = AF_EMA_STEP(sm, e1); sm = AF_EMA_STEP(sm, e2); sm = AF_EMA_STEP(sm, e3);
    }
    for (; x < x1; ++x) sm = AF_EMA_STEP(sm, EB(x));
    return sm;
}
__device__ __forceinline__ uint32_t ema_bits(const float *s_e, uint32_t lead, int x0, uint32_t m, float &sm_io, float alpha, float beta,
                                             float e_min, bool use_smoothed)
{
    float sm = sm_io;
    uint32_t bits = 0, j = 0;
    for (; j + 4 <= m; j += 4) {
        const float e0 = EB(x0 + (int)j), e1 = EB(x0 + (int)j + 1), e2 = EB(x0 + (int)j + 2), e3 = EB(x0 + (int)j + 3);
        sm = AF_EMA_STEP(sm, e0); bits |= ((use_smoothed ? sm : e0) >= e_min ? 1u : 0u) << j;
        sm = AF_EMA_STEP(sm, e1); bits |= ((use_smoothed ? sm : e1) >= e_min ? 1u : 0u) << (j + 1);
        sm = AF_EMA_STEP(sm, e2); bits |= ((use_smoothed ? sm : e2) >= e_min ? 1u : 0u) << (j + 2);
        sm = AF_EMA_STEP(sm, e3); bits |= ((use_smoothed ? sm : e3) >= e_min ? 1u : 0u) << (j + 3);
    }
    for (; j < m; ++j) {
        const float ev = EB(x0 + (int)j);
        sm = AF_EMA_STEP(sm, ev);
        bits |= ((use_smoothed ? sm : ev) >= e_min ? 1u : 0u) << j;
    }
    sm_io = sm;
    return bits;
}

__global__ void __launch_bounds__(SCAN_THREADS) af_vad_scan_par_kernel(const ScanJob J, uint32_t warm)
{
    __shared__ uint32_t s_bits[SCAN_BLOCK / 32];
    __shared__ uint32_t s_entry[SCAN_BLOCK / 32][3];
    __shared__ uint32_t s_exit[SCAN_BLOCK / 32][4];     // per chain head: the machine after the chain, and the OR of its bits
    __shared__ float s_spec[SCAN_BLOCK / SCAN_CHUNK], s_end[SCAN_BLOCK / SCAN_CHUNK];
    __shared__ float s_e[SCAN_E_FLOATS];                // energies of [b0 - lead, b0 + n), padded (epad)
    __shared__ int s_bad;
    const uint32_t s = blockIdx.x, tid = threadIdx.x;
    if (J.recs) {                                        // (uniform over the CTA: before any barrier)
        if (J.recs[s].seq) return;                       // the sequential kernel that follows takes this stream
        warm = J.recs[s].warm;
    }
    const uint32_t T = J.n_frames ? J.n_frames[s] : J.n_frames_all;
    const float *e = J.energy + (uint64_t)s * J.energy_stride;
    uint8_t *out = J.states ? J.states + (uint64_t)s * J.states_stride : nullptr;
    VadState v;
    if (J.state_io) v = J.state_io[s];
    else { v.smoothed = 0.0f; v.state = 0; v.silence_frames = 0; v.speech_frames = 0; }
    const VadParams prm = J.recs ? J.recs[s].prm : J.prm;
    const float alpha = prm.alpha, beta = __fsub_rn(1.0f, prm.alpha), e_min = prm.e_min;
    const bool use_smoothed = alpha > 0.0f;
    const uint32_t timeout = (uint32_t)prm.silence_timeout, minsp = (uint32_t)prm.min_speech;
    // (the host only launches this kernel when every counter fits 32 bits with room to spare)
    float carry_s = v.smoothed;
    VadMachine carry_m{(uint32_t)v.state, (uint32_t)v.silence_frames, (uint32_t)v.speech_frames};
    const bool aligned_out = out && ((reinterpret_cast<uintptr_t>(out) & 15) == 0);

#ifdef AF_SCAN_PROFILE
    long long tp[6]; tp[0] = clock64();
#define AF_SCAN_T(i) tp[i] = clock64();
#else
#define AF_SCAN_T(i)
#endif
    for (uint32_t b0 = 0; b0 < T; b0 += SCAN_BLOCK) {
        const uint32_t n = min(SCAN_BLOCK, T - b0);
        const uint32_t n_chunks = (n + SCAN_CHUNK - 1) / SCAN_CHUNK, n_words = (n + 31) / 32;
        if (tid == 0) s_bad = 0;
        // ---- phase 0: the block's energies and the warm-up before it -> shared memory ----
        const uint32_t lead = min(warm, b0);                 // frames staged in front of the block
#pragma unroll 8
        for (uint32_t i = tid; i < lead + n; i += SCAN_THREADS) s_e[epad(i)] = e[b0 - lead + i];
        __syncthreads();
        AF_SCAN_T(1)
        // ---- phase 1: EMA chunks (speculative start) -> decision bits ----
        for (uint32_t c = tid; c < n_chunks; c += SCAN_THREADS) {
            const uint32_t f_begin = b0 + c * SCAN_CHUNK, f_end = min(f_begin + SCAN_CHUNK, b0 + n);
            float sm;
            if (c == 0) sm = carry_s;
            else {
                // warm-up: from 0 (or, reaching the start of the stream, from the true initial value)
                uint32_t w0;
                if (f_begin >= warm) { w0 = f_begin - warm; sm = 0.0f; }
                else { w0 = 0; sm = v.smoothed; }
                sm = ema_run(s_e, lead, (int)w0 - (int)b0, (int)f_begin - (int)b0, sm, alpha, beta);
                s_spec[c] = sm;
            }
            for (uint32_t f = f_begin; f < f_end; f += 32) {
                const uint32_t m = min(32u, f_end - f);
                s_bits[(f - b0) >> 5] = ema_bits(s_e, lead, (int)(f - b0), m, sm, alpha, beta, e_min, use_smoothed);
            }
            s_end[c] = sm;
        }
        __syncthreads();
        AF_SCAN_T(2)
        // ---- verify every boundary bit for bit ----
        for (uint32_t c = 1 + tid; c < n_chunks; c += SCAN_THREADS)
            if (__float_as_uint(s_spec[c]) != __float_as_uint(s_end[c - 1])) s_bad = 1;
        __syncthreads();
        if (s_bad) {                                      // (rare) redo the block strictly sequentially
            if (tid == 0) {
                float sm = carry_s;
                for (uint32_t w = 0; w < n_words; ++w) {
                    const uint32_t m = min(32u, n - w * 32);
                    uint32_t bits = 0;
                    for (uint32_t j = 0; j < m; ++j) {
                        const float ev = EB(w * 32 + j);
                        sm = __fadd_rn(__fmul_rn(alpha, ev), __fmul_rn(beta, sm));
                        bits |= ((use_smoothed ? sm : ev) >= e_min ? 1u : 0u) << j;
                    }
                    s_bits[w] = bits;
                }
                s_end[n_chunks - 1] = sm;
            }
            __syncthreads();
        }
        AF_SCAN_T(3)
        // ---- phase 2: the machine state at every word boundary ----
        // After `need` = max(timeout, 1) + 1 non-speech frames the machine is in Silence whatever came before (Speech times
        // out, Ending lasts one frame), so a word whose predecessor ends with that many zeros is the head of a CHAIN that can
        // be walked on its own from a fresh Silence; the block's first word starts from the carried state.  One thread per
        // chain (a speech burst and its hang-over: a few words), all chains at once, instead of one thread over all words.
        // What a fresh Silence does not know is the silence_frames count Silence was entered with (it does not act on
        // anything, but it is state): thread 0 hands it down the chains afterwards.
        const uint32_t need = max(timeout, 1u) + 1u;
        if (need <= 32u) {
            for (uint32_t h = tid; h < n_words; h += SCAN_THREADS) {
                if (h != 0u && (s_bits[h - 1] >> (32u - need)) != 0u) continue;         // not a head
                VadMachine m = h == 0u ? carry_m : VadMachine{0u, 0u, 0u};
                EmitNone none;
                uint32_t w = h, seen = 0u;
                for (;;) {
                    const uint32_t bits = s_bits[w], m_n = min(32u, n - w * 32);
                    s_entry[w][0] = m.st; s_entry[w][1] = m.sil; s_entry[w][2] = m.spk;
                    seen |= bits;
                    // whole words of silence in Silence, or of speech in Speech, leave the machine where it is (up to the count)
                    if (m.st == 0u && bits == 0u) {}
                    else if (m.st == 1u && m_n == 32u && bits == 0xffffffffu) { m.spk += 32u; m.sil = 0u; }
                    else vad_machine_word_t(m, bits, m_n, none, timeout, minsp);
                    ++w;
                    if (w >= n_words || (bits >> (32u - need)) == 0u) break;            // the next word heads a chain of its own
                }
                s_exit[h][0] = m.st; s_exit[h][1] = m.sil; s_exit[h][2] = m.spk; s_exit[h][3] = seen;
            }
            __syncthreads();
            if (tid == 0) {
                VadMachine last = carry_m;
                uint32_t w = 0;
                while (w < n_words) {                       // w is a head
                    const uint32_t entry_sil = last.sil;   // true silence_frames at the head (chain 0 already started from it)
                    const bool fresh = w != 0u;
                    uint32_t e = w, seen = 0u;               // patch the words the chain enters in its initial Silence
                    for (;;) {
                        if (fresh && entry_sil != 0u && seen == 0u) s_entry[e][1] = entry_sil;
                        const uint32_t bits = s_bits[e];
                        seen |= bits;
                        ++e;
                        if (e >= n_words || (bits >> (32u - need)) == 0u) break;
                    }
                    last = VadMachine{s_exit[w][0], s_exit[w][1], s_exit[w][2]};
                    if (fresh && s_exit[w][3] == 0u) last.sil = entry_sil;              // never left Silence: the count stays
                    w = e;
                }
                carry_m = last;
            }
        } else if (tid == 0) {
            VadMachine m = carry_m;
            EmitNone none;
            for (uint32_t w = 0; w < n_words; ++w) {
                s_entry[w][0] = m.st; s_entry[w][1] = m.sil; s_entry[w][2] = m.spk;
                vad_machine_word_t(m, s_bits[w], min(32u, n - w * 32), none, timeout, minsp);
            }
            carry_m = m;
        }
        __syncthreads();
        AF_SCAN_T(4)
        // ---- phase 3: every thread expands its words into state bytes ----
        if (out) {
            for (uint32_t w = tid; w < n_words; w += SCAN_THREADS) {
                VadMachine m{s_entry[w][0], s_entry[w][1], s_entry[w][2]};
                EmitMask em;
                const uint32_t m_n = min(32u, n - w * 32);
                vad_machine_word_t(m, s_bits[w], m_n, em, timeout, minsp);
                uint32_t by[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const uint32_t sp = ((em.speech >> (4 * k)) & 0xfu) * 0x00204081u & 0x01010101u;
                    const uint32_t en = ((em.ending >> (4 * k)) & 0xfu) * 0x00204081u & 0x01010101u;
                    by[k] = sp + 2u * en;
                }
                uint8_t *dst = out + b0 + w * 32;
                if (m_n == 32u && aligned_out) {
                    reinterpret_cast<uint4 *>(dst)[0] = make_uint4(by[0], by[1], by[2], by[3]);
                    reinterpret_cast<uint4 *>(dst)[1] = make_uint4(by[4], by[5], by[6], by[7]);
                } else {
#pragma unroll
                    for (int k = 0; k < 8; ++k)
                        for (uint32_t i = 0; i < 4; ++i)
                            if (4u * k + i < m_n) dst[4 * k + i] = (uint8_t)(by[k] >> (8 * i));
                }
            }
        }
        // carries of the next block: the exact EMA value and the machine after the last word
        const float next_s = s_end[n_chunks - 1];
        VadMachine next_m = carry_m;
        if (tid != 0) {
            // recompute the end-of-block machine from the last word's entry (cheap, avoids another broadcast)
            next_m = VadMachine{s_entry[n_words - 1][0], s_entry[n_words - 1][1], s_entry[n_words - 1][2]};
            EmitNone none;
            vad_machine_word_t(next_m, s_bits[n_words - 1], min(32u, n - (n_words - 1) * 32), none, timeout, minsp);
        }
        __syncthreads();                                  // everyone has read s_bits / s_entry / s_end
        carry_s = next_s; carry_m = next_m;
    }
    if (tid == 0) {
        v.smoothed = carry_s; v.state = (int)carry_m.st; v.silence_frames = carry_m.sil; v.speech_frames = carry_m.spk;
        if (J.state_io) J.state_io[s] = v;
        if (J.final_out) J.final_out[s] = v;
    }
#ifdef AF_SCAN_PROFILE
    AF_SCAN_T(5)
    if (tid == 0 && (s == 0 || s == 200)) printf("[scan-profile] stream %u: load %lld  ema %lld  verify %lld  walk %lld  expand %lld cycles\n", s, tp[1] - tp[0], tp[2] - tp[1], tp[3] - tp[2], tp[4] - tp[3], tp[5] - tp[4]);
#endif
}

// ---- long streams: many CTAs per stream ------------------------------------------------------------------------
// The word walk above is sequential per stream (a one-hour recording: 11 250 words through one thread, 2.5 ms).  It is
// cut into blocks of SCAN_BLOCK frames that are walked SPECULATIVELY in parallel, every block but the first assuming a
// fresh machine (Silence, counters 0).  The speculation is exact from the block's first "sync point" on: a speech
// frame that follows at least max(silence_timeout, 1) + 1 non-speech frames finds the machine in Silence whatever came before
// (Speech times out after silence_timeout, Ending lasts one frame) and sets (Speech, 1, 0).  A cheap sequential pass
// then carries the true state from block to block and re-walks only the words in front of each block's sync point
// (the whole block if it has none); the EMA entering a block is speculated from a warm-up and verified the same way.
// Scratch per stream: bits [W], per-word entry states [W][3], per block: spec / end EMA, sync frame, exit state [3].
struct LongScanView {
    uint32_t *bits, *entry;
    float *spec, *end;
    uint32_t *sync, *exit;
};
__host__ __device__ inline uint32_t long_scan_words(uint32_t max_frames) { return (max_frames + 31u) / 32u; }
__host__ __device__ inline uint32_t long_scan_blocks(uint32_t max_frames) { return (max_frames + SCAN_BLOCK - 1u) / SCAN_BLOCK; }
__host__ __device__ inline size_t long_scan_stride(uint32_t max_frames)
{
    return 4 * (size_t)long_scan_words(max_frames) + 6 * (size_t)long_scan_blocks(max_frames);
}
__device__ __forceinline__ LongScanView long_scan_view(uint32_t *scratch, uint32_t max_frames, uint32_t s)
{
    const size_t W = long_scan_words(max_frames), NB = long_scan_blocks(max_frames);
    uint32_t *p = scratch + (size_t)s * long_scan_stride(max_frames);
    LongScanView v;
    v.bits = p; v.entry = p + W;
    v.spec = reinterpret_cast<float *>(p + 4 * W); v.end = v.spec + NB;
    v.sync = p + 4 * W + 2 * NB; v.exit = v.sync + NB;
    return v;
}
size_t scan_scratch_words(uint32_t max_frames) { return long_scan_stride(max_frames); }

constexpr uint32_t NO_SYNC = 0xffffffffu;

// phase A: one CTA per (block, stream): decision bits, speculative walk, sync point, exit state
__global__ void __launch_bounds__(SCAN_THREADS) af_vad_long_a_kernel(const ScanJob J, uint32_t warm)
{
    __shared__ uint32_t s_bits[SCAN_BLOCK / 32];
    __shared__ uint32_t s_exit[SCAN_BLOCK / 32][5];     // per chain head: machine after the chain, OR of its bits, its sync candidate
    __shared__ float s_spec[SCAN_BLOCK / SCAN_CHUNK], s_end[SCAN_BLOCK / SCAN_CHUNK];
    __shared__ float s_e[SCAN_E_FLOATS];
    __shared__ int s_bad;
    const uint32_t blk = blockIdx.x, s = blockIdx.y, tid = threadIdx.x;
    const uint32_t T = J.n_frames ? J.n_frames[s] : J.n_frames_all;
    const uint32_t b0 = blk * SCAN_BLOCK;
    if (b0 >= T) return;
    if (J.recs) {
        if (J.recs[s].seq) return;
        warm = J.recs[s].warm;
    }
    const LongScanView V = long_scan_view(J.scratch, J.max_frames, s);
    const float *e = J.energy + (uint64_t)s * J.energy_stride;
    const VadParams prm = J.recs ? J.recs[s].prm : J.prm;
    const float alpha = prm.alpha, beta = __fsub_rn(1.0f, prm.alpha), e_min = prm.e_min;
    const bool use_smoothed = alpha > 0.0f;
    const uint32_t timeout = (uint32_t)prm.silence_timeout, minsp = (uint32_t)prm.min_speech;
    const uint32_t n = min(SCAN_BLOCK, T - b0);
    const uint32_t n_chunks = (n + SCAN_CHUNK - 1) / SCAN_CHUNK, n_words = (n + 31) / 32;
    if (tid == 0) s_bad = 0;
    const uint32_t lead = min(warm, b0);
#pragma unroll 8
    for (uint32_t i = tid; i < lead + n; i += SCAN_THREADS) s_e[epad(i)] = e[b0 - lead + i];
    __syncthreads();
    // EMA chunks: every chunk but the stream's very first starts from a warm-up (fresh detector: the stream starts at 0)
    for (uint32_t c = tid; c < n_chunks; c += SCAN_THREADS) {
        const uint32_t f_begin = b0 + c * SCAN_CHUNK, f_end = min(f_begin + SCAN_CHUNK, b0 + n);
        float sm = 0.0f;
        if (f_begin != 0) {
            const uint32_t w0 = f_begin >= warm ? f_begin - warm : 0u;
            sm = ema_run(s_e, lead, (int)w0 - (int)b0, (int)f_begin - (int)b0, sm, alpha, beta);
        }
        s_spec[c] = sm;
        for (uint32_t f = f_begin; f < f_end; f += 32) {
            const uint32_t m = min(32u, f_end - f);
            s_bits[(f - b0) >> 5] = ema_bits(s_e, lead, (int)(f - b0), m, sm, alpha, beta, e_min, use_smoothed);
        }
        s_end[c] = sm;
    }
    __syncthreads();
    for (uint32_t c = 1 + tid; c < n_chunks; c += SCAN_THREADS)
        if (__float_as_uint(s_spec[c]) != __float_as_uint(s_end[c - 1])) s_bad = 1;
    __syncthreads();
    if (s_bad && tid == 0) {                                  // (rare) redo the block sequentially from its own start value
        float sm = s_spec[0];
        for (uint32_t w = 0; w < n_words; ++w) {
            const uint32_t m = min(32u, n - w * 32);
            uint32_t bits = 0;
            for (uint32_t j = 0; j < m; ++j) {
                const float ev = EB(w * 32 + j);
                sm = __fadd_rn(__fmul_rn(alpha, ev), __fmul_rn(beta, sm));
                bits |= ((use_smoothed ? sm : ev) >= e_min ? 1u : 0u) << j;
            }
            s_bits[w] = bits;
        }
        s_end[n_chunks - 1] = sm;
    }
    __syncthreads();
    for (uint32_t w = tid; w < n_words; w += SCAN_THREADS) V.bits[(b0 >> 5) + w] = s_bits[w];
    if (tid == 0) { V.spec[blk] = s_spec[0]; V.end[blk] = s_end[n_chunks - 1]; }
    // silence_timeout == 0 behaves like 1 here: the first non-speech frame moves Speech to Ending / Silence, and it takes
    // a second one to leave Ending -- a speech frame right after a single zero would be swallowed by Ending -> Silence
    // (vad.rs:147-151), which a fresh machine does not reproduce
    const uint32_t need = max(timeout, 1u) + 1u;
    if (need <= 32u) {
        // Speculative walk from a fresh machine, chain-parallel as in af_vad_scan_par_kernel: a word whose predecessor ends
        // with `need` non-speech frames heads a chain that starts from a fresh Silence, one thread per chain.  The first speech
        // frame of such a chain is a sync point of the block by construction; inside the block's first chain (which has no
        // run of zeros in front of it) the sync point is searched bit by bit as before.
        for (uint32_t h = tid; h < n_words; h += SCAN_THREADS) {
            if (h != 0u && (s_bits[h - 1] >> (32u - need)) != 0u) continue;             // not a head
            VadMachine m{0u, 0u, 0u};
            EmitNone none;
            uint32_t w = h, seen = 0u, first = NO_SYNC, zrun = 0u;
            for (;;) {
                const uint32_t bits = s_bits[w], m_n = min(32u, n - w * 32);
                uint32_t *en = V.entry + 3 * (size_t)((b0 >> 5) + w);
                en[0] = m.st; en[1] = m.sil; en[2] = m.spk;
                if (h != 0u) {
                    if (first == NO_SYNC && bits != 0u) first = w * 32 + (uint32_t)__ffs((int)bits) - 1u;
                } else if (first == NO_SYNC) {                                      // the block's first chain: bit by bit
                    if (bits == 0u) zrun += m_n;
                    else {
                        for (uint32_t j = 0; j < m_n; ++j) {
                            if ((bits >> j) & 1u) {
                                if (zrun >= need) { first = w * 32 + j; break; }
                                zrun = 0;
                            } else ++zrun;
                        }
                    }
                }
                seen |= bits;
                // whole words of silence in Silence, or of speech in Speech, leave the machine where it is (up to the count)
                if (m.st == 0u && bits == 0u) {}
                else if (m.st == 1u && m_n == 32u && bits == 0xffffffffu) { m.spk += 32u; m.sil = 0u; }
                else vad_machine_word_t(m, bits, m_n, none, timeout, minsp);
                ++w;
                if (w >= n_words || (bits >> (32u - need)) == 0u) break;                // the next word heads a chain of its own
            }
            s_exit[h][0] = m.st; s_exit[h][1] = m.sil; s_exit[h][2] = m.spk; s_exit[h][3] = seen; s_exit[h][4] = first;
        }
        __syncthreads();
        if (tid == 0) {
            // in order over the chains: the block's first sync point, the silence_frames count Silence was entered with (a
            // fresh Silence assumed 0) handed down the chains, the machine after the last one
            VadMachine last{0u, 0u, 0u};
            uint32_t sync = NO_SYNC, w = 0;
            while (w < n_words) {                                                       // w is a head
                const uint32_t entry_sil = last.sil;
                const bool fresh = w != 0u;
                uint32_t e = w, seen = 0u;
                for (;;) {
                    if (fresh && entry_sil != 0u && seen == 0u) V.entry[3 * (size_t)((b0 >> 5) + e) + 1] = entry_sil;
                    const uint32_t bits = s_bits[e];
                    seen |= bits;
                    ++e;
                    if (e >= n_words || (bits >> (32u - need)) == 0u) break;
                }
                if (sync == NO_SYNC) sync = s_exit[w][4];
                last = VadMachine{s_exit[w][0], s_exit[w][1], s_exit[w][2]};
                if (fresh && s_exit[w][3] == 0u) last.sil = entry_sil;                  // never left Silence: the count stays
                w = e;
            }
            V.sync[blk] = sync;
            V.exit[3 * blk] = last.st; V.exit[3 * blk + 1] = last.sil; V.exit[3 * blk + 2] = last.spk;
        }
    } else if (tid == 0) {
        // speculative walk from a fresh machine + the first sync point
        VadMachine m{0u, 0u, 0u};
        EmitNone none;
        uint32_t zrun = 0, sync = NO_SYNC;
        // silence_timeout == 0 behaves like 1 here: the first non-speech frame moves Speech to Ending / Silence, and it takes
        // a second one to leave Ending -- a speech frame right after a single zero would be swallowed by Ending -> Silence
        // (vad.rs:147-151), which a fresh machine does not reproduce
        uint32_t next_bits = s_bits[0];
        for (uint32_t w = 0; w < n_words; ++w) {
            const uint32_t bits = next_bits, m_n = min(32u, n - w * 32);
            if (w + 1 < n_words) next_bits = s_bits[w + 1];                 // (the load overlaps this word's walk)
            uint32_t *en = V.entry + 3 * (size_t)((b0 >> 5) + w);
            en[0] = m.st; en[1] = m.sil; en[2] = m.spk;
            // whole words of silence in Silence, or of speech in Speech, leave the machine where it is (up to the count)
            if (m.st == 0u && bits == 0u) { zrun += m_n; continue; }
            if (m.st == 1u && m_n == 32u && bits == 0xffffffffu && (sync != NO_SYNC || zrun < need)) {
                m.spk += 32u; m.sil = 0u; zrun = 0;
                continue;
            }
            vad_machine_word_t(m, bits, m_n, none, timeout, minsp);
            if (sync == NO_SYNC) {                              // (only until the first one is found)
                if (bits == 0u) zrun += m_n;
                else {
                    for (uint32_t j = 0; j < m_n; ++j) {
                        if ((bits >> j) & 1u) {
                            if (zrun >= need) { sync = w * 32 + j; break; }
                            zrun = 0;
                        } else ++zrun;
                    }
                }
            }
        }
        V.sync[blk] = sync;
        V.exit[3 * blk] = m.st; V.exit[3 * blk + 1] = m.sil; V.exit[3 * blk + 2] = m.spk;
    }
}

// phase B: one WARP per stream carries the true EMA and machine state from block to block.  The walk is sequential, so
// every lane executes it redundantly (same registers, same control flow); what the warp buys is the loads: the per-block
// records of 32 blocks at a time (one per lane, handed round by shuffles) and the decision bits of the words in front of a
// block's sync point as coalesced 32-word loads, instead of a dependent global load per block and per word (33 -> ~10 us
// for one hour of audio).
__global__ void __launch_bounds__(32) af_vad_long_b_kernel(const ScanJob J)
{
    const uint32_t s = blockIdx.x, lane = threadIdx.x;
    if (s >= J.n_streams || (J.recs && J.recs[s].seq)) return;
    const uint32_t T = J.n_frames ? J.n_frames[s] : J.n_frames_all;
    const LongScanView V = long_scan_view(J.scratch, J.max_frames, s);
    const float *e = J.energy + (uint64_t)s * J.energy_stride;
    const VadParams prm = J.recs ? J.recs[s].prm : J.prm;
    const float alpha = prm.alpha, beta = __fsub_rn(1.0f, prm.alpha), e_min = prm.e_min;
    const bool use_smoothed = alpha > 0.0f;
    const uint32_t timeout = (uint32_t)prm.silence_timeout, minsp = (uint32_t)prm.min_speech;
    const uint32_t nb = (T + SCAN_BLOCK - 1) / SCAN_BLOCK;
    constexpr uint32_t FULL = 0xffffffffu;
    float carry_s = 0.0f;
    VadMachine m{0u, 0u, 0u};
    EmitNone none;
    for (uint32_t blk0 = 0; blk0 < nb; blk0 += 32) {
        // the records phase A left for blocks blk0 .. blk0 + 31, one block per lane
        const uint32_t mb = blk0 + lane;
        float l_spec = 0.0f, l_end = 0.0f;
        uint32_t l_sync = NO_SYNC, l_e0 = 0, l_e1 = 0, l_e2 = 0;
        if (mb < nb) {
            l_spec = V.spec[mb]; l_end = V.end[mb]; l_sync = V.sync[mb];
            l_e0 = V.exit[3 * mb]; l_e1 = V.exit[3 * mb + 1]; l_e2 = V.exit[3 * mb + 2];
        }
        const uint32_t kn = min(32u, nb - blk0);
        for (uint32_t k = 0; k < kn; ++k) {
            const uint32_t blk = blk0 + k;
            const float spec = __shfl_sync(FULL, l_spec, k);
            float end_v = __shfl_sync(FULL, l_end, k);
            const uint32_t sync_rec = __shfl_sync(FULL, l_sync, k);
            const VadMachine exit_m{__shfl_sync(FULL, l_e0, k), __shfl_sync(FULL, l_e1, k), __shfl_sync(FULL, l_e2, k)};
            const uint32_t b0 = blk * SCAN_BLOCK, n = min(SCAN_BLOCK, T - b0), n_words = (n + 31) / 32;
            if (blk > 0 && __float_as_uint(spec) != __float_as_uint(carry_s)) {
                // (rare) the warm-up did not reproduce the true EMA: redo this block's decisions from the true value and walk
                // them at once from the true machine state (every lane computes the same; lane 0 stores)
                float sm = carry_s;
                for (uint32_t w = 0; w < n_words; ++w) {
                    const uint32_t mw = min(32u, n - w * 32);
                    uint32_t bits = 0;
                    for (uint32_t j = 0; j < mw; ++j) {
                        const float ev = e[b0 + w * 32 + j];
                        sm = __fadd_rn(__fmul_rn(alpha, ev), __fmul_rn(beta, sm));
                        bits |= ((use_smoothed ? sm : ev) >= e_min ? 1u : 0u) << j;
                    }
                    if (lane == 0) {
                        V.bits[(b0 >> 5) + w] = bits;
                        uint32_t *en = V.entry + 3 * (size_t)((b0 >> 5) + w);
                        en[0] = m.st; en[1] = m.sil; en[2] = m.spk;
                    }
                    vad_machine_word_t(m, bits, mw, none, timeout, minsp);
                }
                if (lane == 0) V.end[blk] = sm;
                carry_s = sm;
                continue;
            }
            carry_s = end_v;
            const bool as_assumed = m.st == 0u && m.sil == 0u && m.spk == 0u;
            if (blk == 0 || as_assumed) {                           // the speculative walk started from the true state
                m = exit_m;
                continue;
            }
            const uint32_t stop = sync_rec == NO_SYNC ? n : sync_rec;   // frames [0, stop) of the block need the true walk
            const uint32_t words = (stop + 31) / 32;
            for (uint32_t w0 = 0; w0 < words; w0 += 32) {
                const uint32_t my = w0 + lane < words ? V.bits[(b0 >> 5) + w0 + lane] : 0u;   // 32 words per load
                const uint32_t wn = min(32u, words - w0);
                for (uint32_t j = 0; j < wn; ++j) {
                    const uint32_t w = w0 + j, bits = __shfl_sync(FULL, my, j);
                    if (lane == 0) {
                        uint32_t *en = V.entry + 3 * (size_t)((b0 >> 5) + w);
                        en[0] = m.st; en[1] = m.sil; en[2] = m.spk;
                    }
                    const uint32_t m_n = min(min(32u, n - w * 32), stop - w * 32);
                    vad_machine_word_t(m, bits, m_n, none, timeout, minsp);
                }
            }
            if (sync_rec != NO_SYNC) m = exit_m;                    // exact from the sync point on
        }
    }
    if (lane == 0) {
        VadState v;
        v.smoothed = carry_s; v.state = (int)m.st; v.silence_frames = m.sil; v.speech_frames = m.spk;
        if (J.final_out) J.final_out[s] = v;
    }
}

// phase C: every word expands into state bytes from its (now exact) entry state
__global__ void __launch_bounds__(SCAN_THREADS) af_vad_long_c_kernel(const ScanJob J)
{
    const uint32_t blk = blockIdx.x, s = blockIdx.y;
    const uint32_t T = J.n_frames ? J.n_frames[s] : J.n_frames_all;
    const uint32_t b0 = blk * SCAN_BLOCK;
    if (b0 >= T || !J.states || (J.recs && J.recs[s].seq)) return;
    const LongScanView V = long_scan_view(J.scratch, J.max_frames, s);
    uint8_t *out = J.states + (uint64_t)s * J.states_stride;
    const bool aligned_out = (reinterpret_cast<uintptr_t>(out) & 15) == 0;
    const VadParams &prm = J.recs ? J.recs[s].prm : J.prm;
    const uint32_t timeout = (uint32_t)prm.silence_timeout, minsp = (uint32_t)prm.min_speech;
    const uint32_t n = min(SCAN_BLOCK, T - b0), n_words = (n + 31) / 32;
    for (uint32_t w = threadIdx.x; w < n_words; w += SCAN_THREADS) {
        const uint32_t *en = V.entry + 3 * (size_t)((b0 >> 5) + w);
        VadMachine m{en[0], en[1], en[2]};
        EmitMask em;
        const uint32_t m_n = min(32u, n - w * 32);
        vad_machine_word_t(m, V.bits[(b0 >> 5) + w], m_n, em, timeout, minsp);
        uint32_t by[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const uint32_t sp = ((em.speech >> (4 * k)) & 0xfu) * 0x00204081u & 0x01010101u;
            const uint32_t en2 = ((em.ending >> (4 * k)) & 0xfu) * 0x00204081u & 0x01010101u;
            by[k] = sp + 2u * en2;
        }
        uint8_t *dst = out + b0 + w * 32;
        if (m_n == 32u && aligned_out) {
            reinterpret_cast<uint4 *>(dst)[0] = make_uint4(by[0], by[1], by[2], by[3]);
            reinterpret_cast<uint4 *>(dst)[1] = make_uint4(by[4], by[5], by[6], by[7]);
        } else {
#pragma unroll
            for (int k = 0; k < 8; ++k)
                for (uint32_t i = 0; i < 4; ++i)
                    if (4u * k + i < m_n) dst[4 * k + i] = (uint8_t)(by[k] >> (8 * i));
        }
    }
}

// warm-up length (frames) after which an EMA started from 0 agrees bit for bit with the true one in practice:
// (1 - alpha)^warm < 2^-56 (24 bits of mantissa + 32 bits of dynamic range); 0 = no parallel scan for this alpha
static uint32_t scan_warmup(float alpha)
{
    if (!(alpha >= 0.0f) || alpha > 1.0f) return 0;       // outside the EMA's sensible range: sequential kernel
    if (alpha == 0.0f || alpha == 1.0f) return 32;        // no memory at all (alpha = 0 never uses the smoothed value)
    const double w = 56.0 / -std::log2(1.0 - (double)alpha);
    if (!(w <= 512.0)) return 0;
    return ((uint32_t)std::ceil(w) + 31u) & ~31u;
}

// the parallel kernel keeps its counters in 32 bits and starts every stream from a fresh detector or from a state the
// caller vouches for; streams resumed from a saved state may hold 64-bit counters -> sequential kernel
static bool scan_small(const VadParams &prm)
{
    return prm.silence_timeout < 0x40000000ull && prm.min_speech < 0x40000000ull;
}

ScanRec scan_rec(const VadParams &prm)
{
    ScanRec r;
    r.prm = prm;
    r.warm = scan_warmup(prm.alpha);
    r.seq = (r.warm == 0 || !scan_small(prm)) ? 1u : 0u;
    return r;
}

// the parallel kernels over all streams of the job (with per-stream records, `warm` is each record's)
static cudaError_t launch_scan_par(const ScanJob &job, uint32_t warm, cudaStream_t st)
{
    if (job.scratch && job.max_frames > 2u * SCAN_BLOCK && job.max_frames < 0x40000000u) {
        // long streams: speculative block walks in parallel, a cheap sequential carry pass, parallel expansion
        const dim3 grid(long_scan_blocks(job.max_frames), job.n_streams);
        af_vad_long_a_kernel<<<grid, SCAN_THREADS, 0, st>>>(job, warm);
        af_vad_long_b_kernel<<<job.n_streams, 32, 0, st>>>(job);
        af_vad_long_c_kernel<<<grid, SCAN_THREADS, 0, st>>>(job);
        return cudaGetLastError();
    }
    af_vad_scan_par_kernel<<<job.n_streams, SCAN_THREADS, 0, st>>>(job, warm);
    return cudaGetLastError();
}

// with per-stream records: does some stream take the parallel kernels?
static bool scan_recs_par(const ScanJob &job)
{
    return job.state_io == nullptr && job.n_frames_all < 0x40000000u && job.n_seq < job.n_streams;
}

uint32_t scan_launches(const ScanJob &job)
{
    return job.recs && scan_recs_par(job) && job.n_seq ? 2u : 1u;
}

cudaError_t launch_vad_scan(const ScanJob &job, cudaStream_t st)
{
    if (job.n_streams == 0) return cudaSuccess;
    const int threads = 32;                       // sequential kernel: one warp per CTA, spread the chains over the SMs
    const uint32_t seq_ctas = (job.n_streams + threads - 1) / threads;
    if (job.recs) {
        // per-stream records: one stream that needs the sequential kernel leaves the others on the parallel ones.  The
        // parallel (or long) kernel runs over all streams and the CTAs of flagged streams exit at once; the sequential
        // kernel follows only when some stream is flagged, and its threads for the other streams exit
        const bool par = scan_recs_par(job);
        if (par) {
            const cudaError_t e = launch_scan_par(job, 0, st);
            if (e != cudaSuccess || job.n_seq == 0) return e;
        }
        af_vad_scan_kernel<<<seq_ctas, threads, 0, st>>>(job, par ? 1u : 0u);
        return cudaGetLastError();
    }
    const uint32_t warm = scan_warmup(job.prm.alpha);
    if (warm != 0 && scan_small(job.prm) && job.n_frames_all < 0x40000000u && job.state_io == nullptr)
        return launch_scan_par(job, warm, st);
    af_vad_scan_kernel<<<seq_ctas, threads, 0, st>>>(job, 0u);
    return cudaGetLastError();
}

// ---- streaming sessions (all streams advance in lockstep) ----
// ingest + resample of one tick in ONE launch: a CTA per stream appends the tick's frames to its input history, then
// resamples the complete chunks out of the row it has just written (the row is read with plain loads after a CTA
// barrier, never through the read-only path); both also carry the retained part of the ping-pong buffers forward,
// skipping what the previous tick consumed (drop / y_drop)
__device__ __forceinline__ float session_resample_one(const SessionResample &J, const float *in, uint32_t i_new)
{
    const unsigned long long n = J.n_begin + i_new;
    if (J.mode == RS_PASSTHROUGH) {
        const long long idx = (long long)n;
        return (idx < J.data_base || idx >= J.n_valid_end) ? 0.0f : in[idx - J.data_base];
    }
    long long k; uint32_t rem;
    resample_pos(n, J.p, J.q, &k, &rem);
    float frac;
    if (J.mode == RS_TABLE) {
        frac = J.frac[i_new];
        k += __float2int_rn((float)rem * (1.0f / (float)J.q) - frac);
    } else {
        frac = (float)rem * (1.0f / (float)J.q);
    }
    float y[4];
#pragma unroll
    for (int t = 0; t < 4; ++t) {
        const long long idx = k - 1 + t;
        y[t] = (idx < J.data_base || idx >= J.n_valid_end) ? 0.0f : in[idx - J.data_base];
    }
    return interp_cubic(frac, y[0], y[1], y[2], y[3]);
}

// zero_history: the 16 retained frames are a fresh stream's zero history; pcm (or nullptr): the new samples also go there
__device__ __forceinline__ void session_tick_row(const SessionIngest &I, const SessionResample &R, uint32_t s, bool zero_history,
                                                 float *pcm)
{
    {
        const float *old = I.old_buf + (uint64_t)s * I.buf_stride;
        float *neu = I.new_buf + (uint64_t)s * I.buf_stride;
        const char *in = reinterpret_cast<const char *>(I.input) + (uint64_t)s * I.in_stride_bytes;
        const uint32_t total = I.keep + I.n_new_frames;
        for (uint32_t i = threadIdx.x; i < total; i += blockDim.x)
            neu[i] = i < I.keep ? (zero_history ? 0.0f : old[I.drop + i])
                                : load_mono(in, I.n_samples, I.n_new_frames, I.channels, I.format, (int)(i - I.keep));
    }
    __syncthreads();                                   // the row written above is read below by other threads of this CTA
    {
        const float *in = R.in_buf + (uint64_t)s * R.in_stride;
        const float *yold = R.y_old + (uint64_t)s * R.y_stride;
        float *ynew = R.y_new + (uint64_t)s * R.y_stride;
        const uint32_t total = R.y_keep + (uint32_t)(R.n_end - R.n_begin);
        if (!pcm) {
            for (uint32_t i = threadIdx.x; i < total; i += blockDim.x)
                ynew[i] = i < R.y_keep ? yold[R.y_drop + i] : session_resample_one(R, in, i - R.y_keep);
        } else {
            for (uint32_t i = threadIdx.x; i < total; i += blockDim.x) {
                if (i < R.y_keep) { ynew[i] = yold[R.y_drop + i]; continue; }
                const float v = session_resample_one(R, in, i - R.y_keep);
                ynew[i] = v;
                pcm[i - R.y_keep] = v;
            }
        }
    }
}

__global__ void __launch_bounds__(256) af_session_tick_kernel(const SessionIngest I, const SessionResample R)
{
    session_tick_row(I, R, blockIdx.x, false, nullptr);
}

cudaError_t launch_session_tick(const SessionIngest &I, const SessionResample &R, uint32_t n_streams, cudaStream_t st)
{
    if (n_streams == 0) return cudaSuccess;
    af_session_tick_kernel<<<n_streams, 256, 0, st>>>(I, R);
    return cudaGetLastError();
}

// independent stream timelines: the same per CTA, with the stream's own lengths and positions from its StreamTick.  A
// restart rewrites the zero history here and clears the stream's detector and wire segment state, so it costs no launch;
// an end's zero padding is never materialised (n_valid_end stops at the data, the reads past it return 0).  Each stream
// takes its channel count and resampling ratio from its format, so one launch serves streams of any mix of formats.
__global__ void __launch_bounds__(256) af_session_tick_streams_kernel(SessionIngest I, SessionResample R, const StreamTick *__restrict__ tab,
                                                                      const SessionFormat *__restrict__ fmts, VadState *vad,
                                                                      uint8_t *wire_prev, float *pcm, uint64_t pcm_stride)
{
    const uint32_t s = blockIdx.x;
    const StreamTick d = tab[s];
    const SessionFormat f = fmts[d.flags >> TICK_FMT_SHIFT];
    I.drop = d.in_drop; I.keep = d.in_keep; I.n_new_frames = d.n_new; I.n_samples = d.n_samples; I.channels = f.channels;
    R.data_base = d.data_base; R.n_valid_end = d.n_valid_end; R.n_begin = d.n_begin; R.n_end = d.n_begin + d.n_y;
    R.frac += d.frac_off; R.y_drop = d.y_drop; R.y_keep = d.y_keep;
    R.p = f.p; R.q = f.q; R.mode = f.mode;
    const bool restart = (d.flags & TICK_RESTART) != 0;
    if (restart && threadIdx.x == 0) {
        VadState v; v.smoothed = 0.0f; v.state = 0; v.silence_frames = 0; v.speech_frames = 0;
        vad[s] = v;
        if (wire_prev) wire_prev[s] = 0;
    }
    session_tick_row(I, R, s, restart, pcm ? pcm + (uint64_t)s * pcm_stride : nullptr);
}

cudaError_t launch_session_tick_streams(const SessionIngest &I, const SessionResample &R, const StreamTick *tab,
                                        const SessionFormat *fmts, VadState *vad, uint8_t *wire_prev, float *pcm,
                                        uint64_t pcm_stride, uint32_t n_streams, cudaStream_t st)
{
    if (n_streams == 0) return cudaSuccess;
    af_session_tick_streams_kernel<<<n_streams, 256, 0, st>>>(I, R, tab, fmts, vad, wire_prev, pcm, pcm_stride);
    return cudaGetLastError();
}

// ---- stream records: one CTA per listed stream gathers (pack) or scatters (unpack) its device state, so that moving a
// whole session costs one launch each way.  The pack writes every byte of the record's device part (zeros past the
// ranges), so two exports of the same state are byte-identical ----
__global__ void __launch_bounds__(128) af_session_pack_kernel(const RecordJob J)
{
    const RecordMove m = J.tab[blockIdx.x];
    uint8_t *r = J.rec + blockIdx.x * J.rec_bytes + J.dev_off;
    float *dst = reinterpret_cast<float *>(r + sizeof(RecordDev));
    const float *in = J.in_buf + (uint64_t)m.slot * J.in_stride + m.in_off;
    const float *y = J.y_buf + (uint64_t)m.slot * J.y_stride + m.y_off;
    for (uint32_t i = threadIdx.x; i < J.n_floats; i += blockDim.x) {
        const uint32_t j = i - REC_IN_FRAMES;
        dst[i] = i < REC_IN_FRAMES ? (i < m.in_len ? in[i] : 0.0f) : (j < m.y_len ? y[j] : 0.0f);
    }
    if (threadIdx.x == 0) {
        RecordDev d;
        d.vad = J.vad[m.slot];
        d.wire = J.wire_prev ? J.wire_prev[m.slot] : 0;
        for (int i = 0; i < 7; ++i) d.pad[i] = 0;
        *reinterpret_cast<RecordDev *>(r) = d;
    }
}

__global__ void __launch_bounds__(128) af_session_unpack_kernel(const RecordJob J)
{
    const RecordMove m = J.tab[blockIdx.x];
    const uint8_t *r = J.rec + blockIdx.x * J.rec_bytes + J.dev_off;
    const float *src = reinterpret_cast<const float *>(r + sizeof(RecordDev));
    float *in = J.in_buf + (uint64_t)m.slot * J.in_stride;
    float *y = J.y_buf + (uint64_t)m.slot * J.y_stride;
    for (uint32_t i = threadIdx.x; i < m.in_len; i += blockDim.x) in[i] = src[i];
    for (uint32_t i = threadIdx.x; i < m.y_len; i += blockDim.x) y[i] = src[REC_IN_FRAMES + i];
    if (threadIdx.x == 0) {
        const RecordDev d = *reinterpret_cast<const RecordDev *>(r);
        J.vad[m.slot] = d.vad;
        if (J.wire_prev) J.wire_prev[m.slot] = m.wire ? d.wire : 0;
    }
}

cudaError_t launch_session_pack(const RecordJob &job, uint32_t n, cudaStream_t st)
{
    if (n == 0) return cudaSuccess;
    af_session_pack_kernel<<<n, 128, 0, st>>>(job);
    return cudaGetLastError();
}

cudaError_t launch_session_unpack(const RecordJob &job, uint32_t n, cudaStream_t st)
{
    if (n == 0) return cudaSuccess;
    af_session_unpack_kernel<<<n, 128, 0, st>>>(job);
    return cudaGetLastError();
}

// ---- level metering (events/mod.rs:41 AudioLevel{level, peak}): peak = max |y| over the tick's new 16 kHz samples ----
// One warp per stream; max is order-independent, so the result is bit-exact against any reference order.
__global__ void af_peak_kernel(const float *__restrict__ y, uint64_t y_stride, uint32_t n, uint32_t n_streams, float *__restrict__ peak,
                               const StreamTick *__restrict__ tab)
{
    const uint32_t s = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (s >= n_streams) return;
    const float *row = y + (uint64_t)s * y_stride;
    if (tab) { row += tab[s].y_keep; n = tab[s].n_y; }
    float m = 0.0f;
    for (uint32_t i = lane; i < n; i += 32) m = fmaxf(m, fabsf(row[i]));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (lane == 0) peak[s] = m;
}

cudaError_t launch_peak(const float *y, uint64_t y_stride, uint32_t n, uint32_t n_streams, float *peak, cudaStream_t st,
                        const StreamTick *tab)
{
    if (n_streams == 0) return cudaSuccess;
    af_peak_kernel<<<(n_streams + 3) / 4, 128, 0, st>>>(y, y_stride, n, n_streams, peak, tab);
    return cudaGetLastError();
}

// ---- f32 -> PCM16 little endian (websocket.rs:246-251): (x.clamp(-1,1) * 32767.0) as i16 ----
__global__ void af_pcm16_kernel(const float *__restrict__ in, uint64_t n, int16_t *__restrict__ out)
{
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        float v = in[i];
        int r = 0;
        if (v == v) {                             // NaN stays NaN through clamp and casts to 0
            v = v < -1.0f ? -1.0f : (v > 1.0f ? 1.0f : v);
            r = __float2int_rz(__fmul_rn(v, 32767.0f));
        }
        out[i] = (int16_t)r;
    }
}

// ---- f32 -> PCM16 LE -> base64 (websocket.rs:244-254): one thread per 3-byte group = 4 characters, one 32-bit store ----
__device__ __forceinline__ uint32_t pcm16_of(float v)
{
    int r = 0;
    if (v == v) {
        v = v < -1.0f ? -1.0f : (v > 1.0f ? 1.0f : v);
        r = __float2int_rz(__fmul_rn(v, 32767.0f));
    }
    return (uint32_t)r & 0xffffu;
}
__device__ __forceinline__ uint32_t b64_char(uint32_t v)      // standard alphabet
{
    return v < 26u ? 'A' + v : (v < 52u ? 'a' + (v - 26u) : (v < 62u ? '0' + (v - 52u) : (v == 62u ? '+' : '/')));
}
// the 4 characters of 3-byte group g of a stream of n_bytes little-endian PCM16 bytes: bytes 3g, 3g+1, 3g+2, where byte k
// is the low (k even) or high half of sample k / 2; a and b are the PCM16 samples 3g / 2 and 3g / 2 + 1 (b = 0 past the end)
__device__ __forceinline__ uint32_t b64_quad(uint32_t a, uint32_t b, uint64_t g, uint64_t n_bytes)
{
    const uint64_t k0 = 3 * g;
    // 32 bits of the stream starting at sample k0 / 2 (little endian), shifted to byte k0
    const uint32_t w = (a | (b << 16)) >> (8 * (uint32_t)(k0 & 1));
    const uint32_t left = (uint32_t)(n_bytes - k0 < 3 ? n_bytes - k0 : 3);          // bytes of this group that exist
    const uint32_t b0 = w & 0xffu, b1 = left > 1 ? (w >> 8) & 0xffu : 0u, b2 = left > 2 ? (w >> 16) & 0xffu : 0u;
    const uint32_t t = (b0 << 16) | (b1 << 8) | b2;
    const uint32_t c0 = b64_char(t >> 18), c1 = b64_char((t >> 12) & 63u);
    const uint32_t c2 = left > 1 ? b64_char((t >> 6) & 63u) : '=', c3 = left > 2 ? b64_char(t & 63u) : '=';
    return c0 | (c1 << 8) | (c2 << 16) | (c3 << 24);
}
__global__ void af_pcm16_base64_kernel(const float *__restrict__ in, uint64_t n, uint32_t *__restrict__ out4)
{
    const uint64_t n_bytes = 2 * n, n_groups = (n_bytes + 2) / 3;
    for (uint64_t g = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; g < n_groups; g += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t s0 = (3 * g) >> 1;
        const uint32_t a = pcm16_of(in[s0]);
        const uint32_t b = s0 + 1 < n ? pcm16_of(in[s0 + 1]) : 0u;
        out4[g] = b64_quad(a, b, g, n_bytes);
    }
}

// ---- session wire output (websocket.rs:244-254 per tick; gated: specs/0001-spec.md:466) ----
// One CTA per stream (grid.x).  Gated, the CTA first lists the tick's kept frames -- the frames of af_vad_segments'
// segments: Speech, or Ending right after Speech -- with ballots and a block scan per 128 frames (T reaches thousands
// with a small custom hop), counting segment starts / closes on the way; payload sample i is then sample
// kept[i / hop] * hop + i % hop of the tick's 16 kHz row.  Ungated, sample i is the tick's new sample i.  Then the PCM16
// row (two samples per 32-bit store), the base64 row (one 3-byte group = 4 characters per 32-bit store) and the record.
// With the segment table on (J.segs), the same rounds list the segment starts with one more ballot: a start's piece begins
// at its position in the kept list, after the piece of the segment open when the tick began (the lead piece, listed first,
// 0 frames when that segment closes on the tick's first frame or by an end without a frame).  A last pass turns the offsets
// into frame counts and marks every piece CLOSED but an open last one.
constexpr uint32_t WIRE_THREADS = 128;
constexpr uint32_t VAD_SPEECH = 1, VAD_ENDING = 2;             // AF_VAD_SPEECH, AF_VAD_ENDING
__device__ __forceinline__ float wire_sample(const WireJob &J, const float *row, const uint16_t *kept, uint32_t y_new, uint32_t i)
{
    return J.gate ? row[(uint32_t)kept[i / J.hop] * J.hop + i % J.hop] : row[y_new + i];
}
// the pieces' frame counts from their offsets (kept: the payload's frames), CLOSED on all but an open last one, the count
__device__ __forceinline__ void wire_segments_close(WireSegment *segs, uint32_t *n_segs, uint32_t np, uint32_t kept,
                                                    bool open)
{
    for (uint32_t i = threadIdx.x; i < np; i += WIRE_THREADS) {
        const uint32_t next = i + 1 < np ? segs[i + 1].offset : kept;
        segs[i].n_frames = next - segs[i].offset;
        if (i + 1 < np || !open) segs[i].flags |= WIRE_SEG_CLOSED;
    }
    if (threadIdx.x == 0) *n_segs = np;
}
__global__ void __launch_bounds__(WIRE_THREADS) af_session_wire_kernel(const WireJob J)
{
    extern __shared__ uint16_t s_kept[];                         // gated: the kept frames of the tick, in order
    __shared__ uint32_t s_warp[WIRE_THREADS / 32];
    __shared__ uint32_t s_wseg[WIRE_THREADS / 32];              // table on: segment starts per warp of the round
    __shared__ uint32_t s_break;                                 // first frame that is not Speech (T if none)
    const uint32_t s = blockIdx.x, t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const float *row = J.y + (uint64_t)s * J.y_stride;
    const uint8_t *st = J.states ? J.states + (uint64_t)s * J.st_stride : nullptr;
    uint32_t T = J.T, y_new = J.y_new, n_new = J.n_new;
    bool end = false;                                            // the stream ends after this tick: an open segment closes
    if (J.tab) { T = J.tab[s].T; y_new = J.tab[s].y_keep; n_new = J.tab[s].n_y; end = (J.tab[s].flags & TICK_END) != 0; }
    if (!st) T = 0;
    const uint32_t prev = J.prev[s];
    WireSegment *segs = J.segs ? J.segs + (uint64_t)s * J.seg_stride : nullptr;
    const uint32_t lead = segs && prev == VAD_SPEECH && (T || end) ? 1u : 0u;   // the open segment's piece comes first
    if (t == 0) {
        s_break = T;
        if (lead) { WireSegment g{}; g.flags = WIRE_SEG_CONTINUED; segs[0] = g; }
    }
    __syncthreads();
    uint32_t kept = 0, started = 0, ended = 0;
    for (uint32_t base = 0; base < T; base += WIRE_THREADS) {   // (uniform trip count: every lane takes the ballots)
        const uint32_t f = base + t;
        const bool valid = f < T;
        const uint32_t cur = valid ? st[f] : 0u, pre = valid ? (f ? st[f - 1] : prev) : 0u;
        const bool sp = cur == VAD_SPEECH, psp = pre == VAD_SPEECH;
        const bool keep = valid && (sp || (cur == VAD_ENDING && psp));
        const bool start = valid && sp && !psp;
        if (valid && !sp) atomicMin(&s_break, f);
        const uint32_t bal = __ballot_sync(0xffffffffu, keep);
        uint32_t sbal = 0;
        if (segs) { sbal = __ballot_sync(0xffffffffu, start); if (lane == 0) s_wseg[warp] = __popc(sbal); }
        if (lane == 0) s_warp[warp] = __popc(bal);
        const uint32_t started0 = started;
        started += __syncthreads_count(start);                   // (the barrier also publishes s_warp, s_wseg)
        ended += __syncthreads_count(valid && psp && !sp);
        uint32_t off = kept, all = 0;
#pragma unroll
        for (uint32_t w = 0; w < WIRE_THREADS / 32; ++w) { off += w < warp ? s_warp[w] : 0u; all += s_warp[w]; }
        off += __popc(bal & ((1u << lane) - 1u));
        if (J.gate && keep) s_kept[off] = (uint16_t)f;
        if (segs && start) {                                     // a start is kept: its piece begins at its payload frame
            uint32_t i = lead + started0 + __popc(sbal & ((1u << lane) - 1u));
#pragma unroll
            for (uint32_t w = 0; w < WIRE_THREADS / 32; ++w) i += w < warp ? s_wseg[w] : 0u;
            WireSegment g{};
            g.frame = (int32_t)f; g.offset = off;
            segs[i] = g;
        }
        kept += all;
        __syncthreads();                                         // s_warp is rewritten by the next round
    }
    if (segs) {
        const bool open = (T ? st[T - 1] : prev) == VAD_SPEECH && !end;
        wire_segments_close(segs, J.n_segs + s, lead + started, kept, open);
    }
    const uint32_t brk = s_break;
    const uint32_t n = J.gate ? kept * J.hop : n_new;
    if (J.pcm16) {
        uint32_t *dst = reinterpret_cast<uint32_t *>(J.pcm16 + (uint64_t)s * J.pcm16_stride);
        for (uint32_t j = t; 2 * j < n; j += WIRE_THREADS) {
            const uint32_t a = pcm16_of(wire_sample(J, row, s_kept, y_new, 2 * j));
            const uint32_t b = 2 * j + 1 < n ? pcm16_of(wire_sample(J, row, s_kept, y_new, 2 * j + 1)) : 0u;
            dst[j] = a | (b << 16);
        }
    }
    const uint32_t n_bytes = 2 * n, n_groups = (n_bytes + 2) / 3;
    if (J.b64) {
        uint32_t *dst = reinterpret_cast<uint32_t *>(J.b64 + (uint64_t)s * J.b64_stride);
        for (uint32_t g = t; g < n_groups; g += WIRE_THREADS) {
            const uint32_t s0 = (3 * g) >> 1;
            const uint32_t a = pcm16_of(wire_sample(J, row, s_kept, y_new, s0));
            const uint32_t b = s0 + 1 < n ? pcm16_of(wire_sample(J, row, s_kept, y_new, s0 + 1)) : 0u;
            dst[g] = b64_quad(a, b, g, n_bytes);
        }
    }
    if (t == 0) {
        // the segment open when the tick began runs on through its Speech frames and the Ending frame closing it
        uint32_t cont = 0;
        if (J.gate && prev == VAD_SPEECH) cont = brk < T ? brk + (st[brk] == VAD_ENDING ? 1u : 0u) : T;
        uint32_t last = T ? st[T - 1] : prev;
        if (end && last == VAD_SPEECH) { ++ended; last = 0; }     // af_vad_segments closes a segment at the last frame
        WireTick r;
        r.n_samples = n; r.n_chars = J.b64 ? 4 * n_groups : 0u; r.continued = cont * J.hop;
        r.started = (uint16_t)started; r.ended = (uint16_t)ended; r.in_speech = last == VAD_SPEECH ? 1 : 0;
        r.pad[0] = r.pad[1] = r.pad[2] = 0;
        J.ticks[s] = r;
        J.prev[s] = (uint8_t)last;
    }
}

// a tick of T frames has at most ceil(T / 2) segment starts (a start follows a frame that is not Speech) and one piece of
// the segment open before it
__host__ __forceinline__ bool wire_segments_fit(const WireSegment *segs, uint64_t stride, uint32_t T)
{
    return !segs || stride >= (uint64_t)(T + 1) / 2 + 1;
}

cudaError_t launch_session_wire(const WireJob &J, cudaStream_t st)
{
    if (J.n_streams == 0) return cudaSuccess;
    if (!wire_segments_fit(J.segs, J.seg_stride, J.states ? J.T : 0)) return cudaErrorInvalidValue;
    const size_t smem = J.gate && J.states ? ((size_t)J.T * sizeof(uint16_t) + 3) & ~(size_t)3 : 0;
    af_session_wire_kernel<<<J.n_streams, WIRE_THREADS, smem, st>>>(J);
    return cudaGetLastError();
}

// ---- session wire features: the log-mel rows of the frames the gated wire payload keeps ----
// One CTA per stream (grid.x), launched before af_session_wire_kernel advances `prev`.  The kept frames are listed by the
// wire kernel's rule (Speech, or Ending right after Speech, the frame before the tick's first being `prev`), written out
// again here so that the wire kernel's code stays as it is; the tests check on every tick that the two agree.  Kept frame
// i's log-mel row then goes to row i of the stream's output: 16-byte loads and stores when rows and strides allow
// (J.vec), else one float per thread.
__global__ void __launch_bounds__(WIRE_THREADS) af_session_wire_logmel_kernel(const WireLogmelJob J)
{
    extern __shared__ uint16_t s_kept[];                         // the kept frames of the tick, in order
    __shared__ uint32_t s_warp[WIRE_THREADS / 32];
    const uint32_t s = blockIdx.x, t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const uint8_t *st = J.states ? J.states + (uint64_t)s * J.st_stride : nullptr;
    uint32_t T = J.tab ? J.tab[s].T : J.T;
    if (!st) T = 0;
    const uint32_t prev = J.prev[s];
    uint32_t kept = 0;
    for (uint32_t base = 0; base < T; base += WIRE_THREADS) {   // (uniform trip count: every lane takes the ballots)
        const uint32_t f = base + t;
        const bool valid = f < T;
        const uint32_t cur = valid ? st[f] : 0u, pre = valid ? (f ? st[f - 1] : prev) : 0u;
        const bool keep = valid && (cur == VAD_SPEECH || (cur == VAD_ENDING && pre == VAD_SPEECH));
        const uint32_t bal = __ballot_sync(0xffffffffu, keep);
        if (lane == 0) s_warp[warp] = __popc(bal);
        __syncthreads();
        uint32_t off = kept, all = 0;
#pragma unroll
        for (uint32_t w = 0; w < WIRE_THREADS / 32; ++w) { off += w < warp ? s_warp[w] : 0u; all += s_warp[w]; }
        if (keep) s_kept[off + __popc(bal & ((1u << lane) - 1u))] = (uint16_t)f;
        kept += all;
        __syncthreads();                                         // s_warp is rewritten by the next round; s_kept is complete
    }
    const uint32_t M = J.n_mels;
    const float *src = J.lm + (uint64_t)s * J.lm_stride;
    float *dst = J.out + (uint64_t)s * J.out_stride;
    if (J.vec) {
        const uint32_t m4 = M / 4, n = kept * m4;
        for (uint32_t i = t; i < n; i += WIRE_THREADS) {
            const uint32_t r = i / m4, c = 4 * (i - r * m4);
            const float4 v = *reinterpret_cast<const float4 *>(src + (uint64_t)s_kept[r] * M + c);
            *reinterpret_cast<float4 *>(dst + (uint64_t)r * M + c) = v;
        }
    } else {
        const uint32_t n = kept * M;
        for (uint32_t i = t; i < n; i += WIRE_THREADS) {
            const uint32_t r = i / M;
            dst[i] = src[(uint64_t)s_kept[r] * M + (i - r * M)];
        }
    }
    if (t == 0) J.n_frames[s] = kept;
}

cudaError_t launch_session_wire_logmel(const WireLogmelJob &J, cudaStream_t st)
{
    if (J.n_streams == 0) return cudaSuccess;
    WireLogmelJob j = J;
    j.vec = J.n_mels % 4 == 0 && J.lm_stride % 4 == 0 && J.out_stride % 4 == 0 &&
            ((reinterpret_cast<uintptr_t>(J.lm) | reinterpret_cast<uintptr_t>(J.out)) & 15) == 0;
    const size_t smem = J.states ? ((size_t)J.T * sizeof(uint16_t) + 3) & ~(size_t)3 : 0;
    af_session_wire_logmel_kernel<<<J.n_streams, WIRE_THREADS, smem, st>>>(j);
    return cudaGetLastError();
}

// ---- session wire pre-roll: every segment the gated payload starts reaches back up to P frames ----
// One CTA per stream (grid.x), launched after the scan instead of the features and wire kernels.  Frames are numbered
// virtually: v < h is the v-th oldest of the h history frames (the frames after the stream's last kept frame, since its
// origin, at most P), v >= h is the tick's frame v - h.  A kept frame's predecessor is kept unless it starts a segment, so
// a frame is in the payload exactly when a kept frame of the tick lies within [v, v + P]: the kept frames themselves and
// the pre-roll of every segment start, clamped at the previous kept frame and the origin by what the history holds.
// (1) the kept bits and the events, by the wire kernel's rule; (2) the payload's frames, ballots and a block scan;
// (3) PCM16, base64, log-mel rows and the record, pre-roll frames of earlier pushes read from the history; (4) after a
// barrier, the tick's frames after its last kept frame (all of them if none is kept) go into the history.
// Table on (J.segs): in (2) a payload frame begins a piece when it is a pre-roll frame or a segment start and the payload
// frame before it, if any, is not adjacent or is kept: everything between a kept frame and the next start belongs to the
// start's pre-roll.  The lead piece (the segment open when the tick began) comes first, as in the wire kernel.
__device__ __forceinline__ bool any_kept(const uint32_t *bits, int32_t lo, int32_t hi)   // a kept frame in [lo, hi)?
{
    if (lo >= hi) return false;
    const uint32_t w0 = (uint32_t)lo >> 5, w1 = (uint32_t)(hi - 1) >> 5;
    for (uint32_t w = w0; w <= w1; ++w) {
        uint32_t b = bits[w];
        if (w == w0) b &= 0xffffffffu << (lo & 31);
        if (w == w1) b &= 0xffffffffu >> (31 - ((hi - 1) & 31));
        if (b) return true;
    }
    return false;
}
// first kept frame in [lo, hi), or hi
__device__ __forceinline__ int32_t first_kept(const uint32_t *bits, int32_t lo, int32_t hi)
{
    while (lo < hi) {
        const uint32_t b = bits[lo >> 5] & (0xffffffffu << (lo & 31));
        if (b) return min((lo & ~31) + __ffs(b) - 1, hi);
        lo = (lo & ~31) + 32;
    }
    return hi;
}
// payload sample i as PCM16: history frames were stored encoded, tick frames are encoded here (head: the ring slot of
// the oldest history frame)
__device__ __forceinline__ uint32_t preroll_sample(const WirePrerollJob &J, const float *row, const int16_t *hist,
                                                   const uint16_t *list, uint32_t h, uint32_t head, uint32_t i)
{
    const uint32_t v = list[i / J.hop], j = i % J.hop;
    if (v < h) return (uint32_t)(uint16_t)hist[((head + v) % J.P) * J.hop + j];
    return pcm16_of(row[(v - h) * J.hop + j]);
}
__global__ void __launch_bounds__(WIRE_THREADS) af_session_wire_preroll_kernel(const WirePrerollJob J)
{
    extern __shared__ uint32_t s_dyn[];
    const uint32_t n_words = (J.T + 31) / 32;
    uint32_t *s_bits = s_dyn;                                    // bit f % 32 of word f / 32: tick frame f is kept
    uint16_t *s_list = reinterpret_cast<uint16_t *>(s_dyn + n_words);   // the payload's frames, virtual, in order
    __shared__ uint32_t s_warp[WIRE_THREADS / 32];
    __shared__ uint32_t s_wseg[WIRE_THREADS / 32];              // table on: pieces begun per warp of the round
    __shared__ uint32_t s_break;                                 // first frame that is not Speech (T if none)
    __shared__ int32_t s_last;                                   // last kept frame of the tick (-1 if none)
    const uint32_t s = blockIdx.x, t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const float *row = J.y + (uint64_t)s * J.y_stride;
    const uint8_t *st = J.states ? J.states + (uint64_t)s * J.st_stride : nullptr;
    uint32_t T = J.T;
    bool end = false, restart = false;
    if (J.tab) { T = J.tab[s].T; end = (J.tab[s].flags & TICK_END) != 0; restart = (J.tab[s].flags & TICK_RESTART) != 0; }
    if (!st) T = 0;
    const uint32_t prev = J.prev[s], P = J.P, hop = J.hop;
    const uint32_t h = restart ? 0u : J.hist_n[s], pos = J.hist_pos[s];
    const uint32_t head = (pos + P - h) % P;
    WireSegment *segs = J.segs ? J.segs + (uint64_t)s * J.seg_stride : nullptr;
    const uint32_t lead = segs && prev == VAD_SPEECH && (T || end) ? 1u : 0u;   // the open segment's piece comes first
    if (t == 0) {
        s_break = T; s_last = -1;
        if (lead) { WireSegment g{}; g.flags = WIRE_SEG_CONTINUED; segs[0] = g; }
    }
    __syncthreads();
    uint32_t started = 0, ended = 0;
    for (uint32_t base = 0; base < T; base += WIRE_THREADS) {   // (uniform trip count: every lane takes the ballots)
        const uint32_t f = base + t;
        const bool valid = f < T;
        const uint32_t cur = valid ? st[f] : 0u, pre = valid ? (f ? st[f - 1] : prev) : 0u;
        const bool sp = cur == VAD_SPEECH, psp = pre == VAD_SPEECH;
        const bool keep = valid && (sp || (cur == VAD_ENDING && psp));
        if (valid && !sp) atomicMin(&s_break, f);
        if (keep) atomicMax(&s_last, (int32_t)f);
        const uint32_t bal = __ballot_sync(0xffffffffu, keep);
        const uint32_t w = (base >> 5) + warp;
        if (lane == 0 && w < n_words) s_bits[w] = bal;
        started += __syncthreads_count(valid && sp && !psp);    // (the barriers also publish s_bits, s_last, s_break)
        ended += __syncthreads_count(valid && psp && !sp);
    }
    const uint32_t V = h + T;
    uint32_t n_list = 0, n_pieces = lead;
    for (uint32_t base = 0; base < V; base += WIRE_THREADS) {
        const uint32_t v = base + t;
        const int32_t f = (int32_t)v - (int32_t)h;
        const bool in = v < V && any_kept(s_bits, max(f, 0), min(f + (int32_t)P + 1, (int32_t)T));
        const uint32_t bal = __ballot_sync(0xffffffffu, in);
        if (lane == 0) s_warp[warp] = __popc(bal);
        bool begins = false, kept_v = false;
        uint32_t pbal = 0;
        if (segs) {
            if (in) {                                            // (then f < T)
                kept_v = f >= 0 && ((s_bits[f >> 5] >> (f & 31)) & 1u);
                const bool start = kept_v && st[f] == VAD_SPEECH && (f ? st[f - 1] : prev) != VAD_SPEECH;
                const bool kept_p = f >= 1 && ((s_bits[(f - 1) >> 5] >> ((f - 1) & 31)) & 1u);
                begins = (start || !kept_v) &&
                         (v == 0 || kept_p || !any_kept(s_bits, max(f - 1, 0), min(f + (int32_t)P, (int32_t)T)));
            }
            pbal = __ballot_sync(0xffffffffu, begins);
            if (lane == 0) s_wseg[warp] = __popc(pbal);
        }
        __syncthreads();
        uint32_t off = n_list, all = 0;
#pragma unroll
        for (uint32_t w = 0; w < WIRE_THREADS / 32; ++w) { off += w < warp ? s_warp[w] : 0u; all += s_warp[w]; }
        off += __popc(bal & ((1u << lane) - 1u));
        if (in) s_list[off] = (uint16_t)v;
        if (segs) {
            uint32_t i = n_pieces + __popc(pbal & ((1u << lane) - 1u)), pieces = 0;
#pragma unroll
            for (uint32_t w = 0; w < WIRE_THREADS / 32; ++w) { i += w < warp ? s_wseg[w] : 0u; pieces += s_wseg[w]; }
            if (begins) {                                        // a pre-roll frame's onset is the first kept frame after it
                WireSegment g{};
                g.frame = f; g.offset = off;
                g.preroll = kept_v ? 0 : (uint16_t)(first_kept(s_bits, max(f, 0), min(f + (int32_t)P + 1, (int32_t)T)) - f);
                segs[i] = g;
            }
            n_pieces += pieces;
        }
        n_list += all;
        __syncthreads();                                         // s_warp is rewritten by the next round; s_list is complete
    }
    if (segs) {
        const bool open = (T ? st[T - 1] : prev) == VAD_SPEECH && !end;
        wire_segments_close(segs, J.n_segs + s, n_pieces, n_list, open);
    }
    const int16_t *hist = J.hist_pcm + (uint64_t)s * P * hop;
    const uint32_t n = n_list * hop;
    if (J.pcm16) {
        uint32_t *dst = reinterpret_cast<uint32_t *>(J.pcm16 + (uint64_t)s * J.pcm16_stride);
        for (uint32_t j = t; 2 * j < n; j += WIRE_THREADS) {
            const uint32_t a = preroll_sample(J, row, hist, s_list, h, head, 2 * j);
            const uint32_t b = 2 * j + 1 < n ? preroll_sample(J, row, hist, s_list, h, head, 2 * j + 1) : 0u;
            dst[j] = a | (b << 16);
        }
    }
    const uint32_t n_bytes = 2 * n, n_groups = (n_bytes + 2) / 3;
    if (J.b64) {
        uint32_t *dst = reinterpret_cast<uint32_t *>(J.b64 + (uint64_t)s * J.b64_stride);
        for (uint32_t g = t; g < n_groups; g += WIRE_THREADS) {
            const uint32_t s0 = (3 * g) >> 1;
            const uint32_t a = preroll_sample(J, row, hist, s_list, h, head, s0);
            const uint32_t b = s0 + 1 < n ? preroll_sample(J, row, hist, s_list, h, head, s0 + 1) : 0u;
            dst[g] = b64_quad(a, b, g, n_bytes);
        }
    }
    const uint32_t M = J.n_mels;
    if (J.lm_out) {
        const float *src = J.lm + (uint64_t)s * J.lm_stride, *hl = J.hist_lm + (uint64_t)s * P * M;
        float *dst = J.lm_out + (uint64_t)s * J.lm_out_stride;
        for (uint32_t i = t; i < n_list * M; i += WIRE_THREADS) {
            const uint32_t r = i / M, c = i - r * M, v = s_list[r];
            dst[i] = v < h ? hl[((head + v) % P) * M + c] : src[(uint64_t)(v - h) * M + c];
        }
    }
    if (t == 0) {
        // the wire kernel's record; only n_samples and n_chars count the pre-roll
        uint32_t cont = 0;
        if (prev == VAD_SPEECH) cont = s_break < T ? s_break + (st[s_break] == VAD_ENDING ? 1u : 0u) : T;
        uint32_t last = T ? st[T - 1] : prev;
        if (end && last == VAD_SPEECH) { ++ended; last = 0; }
        WireTick r;
        r.n_samples = n; r.n_chars = J.b64 ? 4 * n_groups : 0u; r.continued = cont * hop;
        r.started = (uint16_t)started; r.ended = (uint16_t)ended; r.in_speech = last == VAD_SPEECH ? 1 : 0;
        r.pad[0] = r.pad[1] = r.pad[2] = 0;
        J.ticks[s] = r;
        J.prev[s] = (uint8_t)last;
        if (J.lm_out) J.n_frames[s] = n_list;
    }
    __syncthreads();                                             // every history read above is done
    const int32_t lk = s_last;
    const uint32_t n_app = T - (uint32_t)(lk + 1), skip = n_app > P ? n_app - P : 0u;
    if (!end) {                                                  // (an end empties the history: the next push is an origin)
        int16_t *hp = J.hist_pcm + (uint64_t)s * P * hop;
        for (uint32_t i = t; i < (n_app - skip) * hop; i += WIRE_THREADS) {
            const uint32_t j = skip + i / hop, k = i % hop;
            hp[((pos + j) % P) * hop + k] = (int16_t)pcm16_of(row[(uint64_t)(lk + 1 + j) * hop + k]);
        }
        if (J.lm_out) {
            const float *src = J.lm + (uint64_t)s * J.lm_stride;
            float *hl = J.hist_lm + (uint64_t)s * P * M;
            for (uint32_t i = t; i < (n_app - skip) * M; i += WIRE_THREADS) {
                const uint32_t j = skip + i / M, c = i % M;
                hl[((pos + j) % P) * M + c] = src[(uint64_t)(lk + 1 + j) * M + c];
            }
        }
    }
    if (t == 0) {
        J.hist_n[s] = end ? 0u : min(P, (lk >= 0 ? 0u : h) + n_app);
        J.hist_pos[s] = (pos + n_app) % P;
    }
}

cudaError_t launch_session_wire_preroll(const WirePrerollJob &J, cudaStream_t st)
{
    if (J.n_streams == 0) return cudaSuccess;
    const size_t smem = (size_t)(J.T + 31) / 32 * sizeof(uint32_t) + (((size_t)(J.T + J.P) * sizeof(uint16_t) + 3) & ~(size_t)3);
    if (J.T + J.P > 0xffffu) return cudaErrorInvalidValue;      // (frame indices are 16-bit, as in the wire kernel)
    if (!wire_segments_fit(J.segs, J.seg_stride, J.states ? J.T : 0)) return cudaErrorInvalidValue;
    if (smem > 48 * 1024) {
        const cudaError_t e = cudaFuncSetAttribute(af_session_wire_preroll_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    af_session_wire_preroll_kernel<<<J.n_streams, WIRE_THREADS, smem, st>>>(J);
    return cudaGetLastError();
}

__global__ void af_session_preroll_clear_kernel(const RecordMove *__restrict__ tab, uint32_t n, uint32_t *__restrict__ hist_n)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) hist_n[tab[i].slot] = 0;
}

cudaError_t launch_session_preroll_clear(const RecordMove *tab, uint32_t n, uint32_t *hist_n, cudaStream_t st)
{
    if (n == 0) return cudaSuccess;
    af_session_preroll_clear_kernel<<<(n + 255) / 256, 256, 0, st>>>(tab, n, hist_n);
    return cudaGetLastError();
}

// the same over the rows of a batch: in [rows][in_stride] f32 -> out [rows][out_stride] i16, `width` samples per row
// (four at a time: one 16-byte load, one 8-byte store; both strides are multiples of 4)
__global__ void af_pcm16_rows_kernel(const float *__restrict__ in, uint64_t in_stride, int16_t *__restrict__ out, uint64_t out_stride,
                                     uint32_t width)
{
    const float4 *row = reinterpret_cast<const float4 *>(in + (uint64_t)blockIdx.y * in_stride);
    uint2 *dst = reinterpret_cast<uint2 *>(out + (uint64_t)blockIdx.y * out_stride);
    const uint32_t n4 = (width + 3) / 4;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += gridDim.x * blockDim.x) {
        const float4 v = __ldcs(row + i);
        const float f[4] = {v.x, v.y, v.z, v.w};
        int r[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            float x = f[k];
            r[k] = 0;
            if (x == x) {
                x = x < -1.0f ? -1.0f : (x > 1.0f ? 1.0f : x);
                r[k] = __float2int_rz(__fmul_rn(x, 32767.0f));
            }
        }
        __stcs(dst + i, make_uint2(((uint32_t)r[0] & 0xffffu) | ((uint32_t)r[1] << 16), ((uint32_t)r[2] & 0xffffu) | ((uint32_t)r[3] << 16)));
    }
}

cudaError_t launch_pcm16_rows(const float *in, uint64_t in_stride, int16_t *out, uint64_t out_stride, uint32_t width, uint32_t rows,
                              cudaStream_t st)
{
    if (rows == 0 || width == 0) return cudaSuccess;
    const uint32_t gx = std::max<uint32_t>(1u, std::min<uint32_t>((width / 4 + 255) / 256, (8u * 148u + rows - 1) / rows));
    af_pcm16_rows_kernel<<<dim3(gx, rows), 256, 0, st>>>(in, in_stride, out, out_stride, width);
    return cudaGetLastError();
}

cudaError_t launch_pcm16(const float *in, uint64_t n, int16_t *out, cudaStream_t st)
{
    if (n == 0) return cudaSuccess;
    const int blocks = (int)std::min<uint64_t>((n + 255) / 256, 148 * 8);
    af_pcm16_kernel<<<blocks, 256, 0, st>>>(in, n, out);
    return cudaGetLastError();
}

cudaError_t launch_pcm16_base64(const float *in, uint64_t n, char *out, cudaStream_t st)
{
    if (n == 0) return cudaSuccess;
    const uint64_t groups = (2 * n + 2) / 3;
    const int blocks = (int)std::min<uint64_t>((groups + 255) / 256, 148 * 8);
    af_pcm16_base64_kernel<<<blocks, 256, 0, st>>>(in, n, reinterpret_cast<uint32_t *>(out));
    return cudaGetLastError();
}

// ---- VAD segmentation: runs from the first Speech frame to Ending (inclusive) / Silence (exclusive) ----
// One CTA per stream.  A segment starts at every frame with state Speech whose predecessor is not Speech, and
// ends at the first later frame that is not Speech; starts and ends alternate, so the k-th start pairs with
// the k-th end.  Each thread owns a contiguous span of frames (a multiple of 16, read 16 states per load and
// turned into a 16-bit "is Speech" mask): count, block-wide exclusive scan, write.
constexpr uint32_t SEG_THREADS = 1024;
__device__ __forceinline__ uint32_t speech_mask16(const uint8_t *st, uint32_t f, uint32_t T, bool vec)
{
    // bit i: frame f + i is Speech (frames >= T read as not Speech)
    uint32_t m = 0;
    if (vec && f + 16 <= T) {
        const uint4 v = *reinterpret_cast<const uint4 *>(st + f);
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const uint32_t eq = __vcmpeq4(w[k], 0x01010101u) & 0x01010101u;        // 1 per Speech byte
            m |= (((eq * 0x01020408u) >> 24) & 0xfu) << (4 * k);                     // gather the four flags (byte i -> bit i)
        }
    } else {
        for (uint32_t i = 0; i < 16 && f + i < T; ++i) m |= (st[f + i] == 1 ? 1u : 0u) << i;
    }
    return m;
}
__global__ void __launch_bounds__(SEG_THREADS) af_vad_segments_kernel(const uint8_t *__restrict__ states, uint64_t stride,
                                                                      const uint32_t *__restrict__ n_frames, uint32_t n_streams,
                                                                      uint32_t *__restrict__ seg, uint32_t seg_cap,
                                                                      uint32_t *__restrict__ n_seg)
{
    __shared__ uint32_t s_starts[SEG_THREADS], s_ends[SEG_THREADS];
    const uint32_t s = blockIdx.x;
    if (s >= n_streams) return;
    const uint8_t *st = states + (uint64_t)s * stride;
    uint32_t *sg = seg + (uint64_t)s * seg_cap * 2;
    const uint32_t T = n_frames[s];
    const uint32_t nt = blockDim.x, t = threadIdx.x;
    const bool vec = (reinterpret_cast<uintptr_t>(st) & 15) == 0;
    const uint32_t span = (((T + nt - 1) / nt) + 15u) & ~15u;           // frames per thread, a multiple of 16
    const uint32_t lo = min(t * span, T), hi = min(lo + span, T);
    uint32_t ns = 0, ne = 0;
    uint32_t prev = lo > 0 ? (st[lo - 1] == 1 ? 1u : 0u) : 0u;
    for (uint32_t f = lo; f < hi; f += 16) {
        const uint32_t m = speech_mask16(st, f, hi, vec), n = min(16u, hi - f);
        const uint32_t before = ((m << 1) | prev) & 0xffffu;            // bit i: frame f + i - 1 is Speech
        const uint32_t valid = n >= 16 ? 0xffffu : ((1u << n) - 1u);
        ns += __popc(m & ~before & valid);
        ne += __popc(~m & before & valid);
        prev = (m >> (n - 1)) & 1u;
    }
    s_starts[t] = ns; s_ends[t] = ne;
    __syncthreads();
    // exclusive scan (Hillis-Steele on both arrays)
    for (uint32_t d = 1; d < nt; d <<= 1) {
        uint32_t a = 0, b = 0;
        if (t >= d) { a = s_starts[t - d]; b = s_ends[t - d]; }
        __syncthreads();
        s_starts[t] += a; s_ends[t] += b;
        __syncthreads();
    }
    uint32_t ks = s_starts[t] - ns, ke = s_ends[t] - ne;      // index of this span's first start / end
    const uint32_t total = s_starts[nt - 1], total_ends = s_ends[nt - 1];
    if (ns | ne) {                                            // only spans with a boundary take the second pass
        prev = lo > 0 ? (st[lo - 1] == 1 ? 1u : 0u) : 0u;
        for (uint32_t f = lo; f < hi; f += 16) {
            const uint32_t m = speech_mask16(st, f, hi, vec), n = min(16u, hi - f);
            const uint32_t before = ((m << 1) | prev) & 0xffffu;
            const uint32_t valid = n >= 16 ? 0xffffu : ((1u << n) - 1u);
            uint32_t sb = m & ~before & valid, eb = ~m & before & valid;
            while (sb) { const uint32_t i = __ffs((int)sb) - 1u; sb &= sb - 1u; if (ks < seg_cap) sg[2 * ks] = f + i; ks++; }
            while (eb) {
                const uint32_t i = __ffs((int)eb) - 1u; eb &= eb - 1u;
                if (ke < seg_cap) sg[2 * ke + 1] = st[f + i] == 2 ? f + i + 1 : f + i;     // Ending belongs to the segment
                ke++;
            }
            prev = (m >> (n - 1)) & 1u;
        }
    }
    if (t == 0) {
        if (total > total_ends && total - 1 < seg_cap) sg[2 * (total - 1) + 1] = T;    // still speaking at the end
        n_seg[s] = total;
    }
}

cudaError_t launch_vad_segments(const uint8_t *states, uint64_t stride, const uint32_t *n_frames, uint32_t n_streams,
                                uint32_t *seg, uint32_t seg_cap, uint32_t *n_seg, cudaStream_t st)
{
    if (n_streams == 0) return cudaSuccess;
    af_vad_segments_kernel<<<n_streams, SEG_THREADS, 0, st>>>(states, stride, n_frames, n_streams, seg, seg_cap, n_seg);
    return cudaGetLastError();
}

// ---- segment pre-roll: one thread per segment slot.  A thread rewrites its segment's start and reads only the end of
// the one before, so the update in place has no hazard ----
__global__ void af_vad_segments_preroll_kernel(uint32_t *__restrict__ seg, uint32_t seg_cap, const uint32_t *__restrict__ n_seg,
                                               uint32_t n_streams, uint32_t P)
{
    const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= (uint64_t)n_streams * seg_cap) return;
    const uint32_t s = (uint32_t)(i / seg_cap), k = (uint32_t)(i - (uint64_t)s * seg_cap);
    if (k >= n_seg[s]) return;
    uint32_t *sg = seg + 2 * i;
    const uint32_t start = sg[0], lo = k ? sg[-1] : 0u;         // the previous segment's end (exclusive), or frame 0
    sg[0] = max(start > P ? start - P : 0u, min(lo, start));
}

cudaError_t launch_vad_segments_preroll(uint32_t *seg, uint32_t seg_cap, const uint32_t *n_seg, uint32_t n_streams, uint32_t P,
                                        cudaStream_t st)
{
    const uint64_t n = (uint64_t)n_streams * seg_cap;
    if (n == 0 || P == 0) return cudaSuccess;
    af_vad_segments_preroll_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(seg, seg_cap, n_seg, n_streams, P);
    return cudaGetLastError();
}

// ---- VAD-gated output (SURVEY 8(f) f1; intent: specs/0001-spec.md:466 "filter the silent stretches before sending") ----
// The segments [start, end) of a stream select the frames whose audio is kept: frame f contributes its hop, samples
// [f hop, (f + 1) hop), and its log-mel row.  The kept frames of a stream are packed in order; segment k starts at
// compacted frame off[k] = sum of the lengths of the segments before it (off[n_seg] = total).
// (1) offsets: one CTA per stream, block-wide exclusive scan of the segment lengths.
constexpr uint32_t GATE_THREADS = 256;
__global__ void __launch_bounds__(GATE_THREADS) af_gate_offsets_kernel(const uint32_t *__restrict__ seg, uint32_t seg_cap,
                                                                       const uint32_t *__restrict__ n_seg, uint32_t *__restrict__ off,
                                                                       uint32_t *__restrict__ total)
{
    __shared__ uint32_t s_part[GATE_THREADS];
    const uint32_t s = blockIdx.x, t = threadIdx.x;
    const uint32_t n = min(n_seg[s], seg_cap);
    const uint32_t *sg = seg + (uint64_t)s * seg_cap * 2;
    uint32_t *of = off + (uint64_t)s * (seg_cap + 1);
    const uint32_t per = (n + GATE_THREADS - 1) / GATE_THREADS;
    const uint32_t lo = min(t * per, n), hi = min(lo + per, n);
    uint32_t sum = 0;
    for (uint32_t k = lo; k < hi; ++k) sum += sg[2 * k + 1] - sg[2 * k];
    s_part[t] = sum;
    __syncthreads();
    for (uint32_t d = 1; d < GATE_THREADS; d <<= 1) {
        const uint32_t a = t >= d ? s_part[t - d] : 0u;
        __syncthreads();
        s_part[t] += a;
        __syncthreads();
    }
    uint32_t run = s_part[t] - sum;
    for (uint32_t k = lo; k < hi; ++k) { of[k] = run; run += sg[2 * k + 1] - sg[2 * k]; }
    if (t == GATE_THREADS - 1) { of[n] = s_part[t]; total[s] = s_part[t]; }
}
// (2) copy: one warp per compacted frame (binary search of its segment, then 16-byte copies of its hop of PCM and its
// log-mel row); grid.y = stream, the warps of grid.x stride over the stream's compacted frames
__global__ void __launch_bounds__(GATE_THREADS) af_gate_copy_kernel(const float *__restrict__ pcm, uint64_t pcm_stride,
                                                                    const float *__restrict__ logmel, uint64_t logmel_stride,
                                                                    uint32_t n_mels, const uint32_t *__restrict__ n_out, uint32_t hop,
                                                                    const uint32_t *__restrict__ seg, uint32_t seg_cap,
                                                                    const uint32_t *__restrict__ n_seg, const uint32_t *__restrict__ off,
                                                                    float *__restrict__ out_pcm, uint64_t out_pcm_stride,
                                                                    float *__restrict__ out_lm, uint64_t out_lm_stride)
{
    const uint32_t s = blockIdx.y, lane = threadIdx.x & 31;
    const uint32_t n = min(n_seg[s], seg_cap);
    const uint32_t *sg = seg + (uint64_t)s * seg_cap * 2;
    const uint32_t *of = off + (uint64_t)s * (seg_cap + 1);
    const uint32_t total = of[n];
    const uint32_t n_samples = n_out ? n_out[s] : 0xffffffffu;
    const float *src_p = pcm ? pcm + (uint64_t)s * pcm_stride : nullptr;
    float *dst_p = out_pcm ? out_pcm + (uint64_t)s * out_pcm_stride : nullptr;
    const float *src_l = logmel ? logmel + (uint64_t)s * logmel_stride : nullptr;
    float *dst_l = out_lm ? out_lm + (uint64_t)s * out_lm_stride : nullptr;
    const bool vec_p = (hop & 3u) == 0 && ((reinterpret_cast<uintptr_t>(src_p) | reinterpret_cast<uintptr_t>(dst_p)) & 15) == 0;
    const bool vec_l = (n_mels & 3u) == 0 && ((reinterpret_cast<uintptr_t>(src_l) | reinterpret_cast<uintptr_t>(dst_l)) & 15) == 0;
    const uint32_t warps = gridDim.x * (GATE_THREADS / 32);
    for (uint32_t j = blockIdx.x * (GATE_THREADS / 32) + (threadIdx.x >> 5); j < total; j += warps) {
        uint32_t a = 0, b = n;                               // largest k with off[k] <= j (segments are never empty)
        while (b - a > 1) { const uint32_t m = (a + b) >> 1; if (of[m] <= j) a = m; else b = m; }
        const uint32_t f = sg[2 * a] + (j - of[a]);          // source frame
        if (src_p && dst_p) {
            const uint64_t so = (uint64_t)f * hop, dof = (uint64_t)j * hop;
            const uint32_t cnt = so >= n_samples ? 0u : (uint32_t)min((uint64_t)hop, (uint64_t)n_samples - so);
            if (vec_p && cnt == hop) {
                const float4 *sp = reinterpret_cast<const float4 *>(src_p + so);
                float4 *dp = reinterpret_cast<float4 *>(dst_p + dof);
                for (uint32_t i = lane; i < hop / 4; i += 32) __stcs(dp + i, __ldcs(sp + i));
            } else {
                for (uint32_t i = lane; i < hop; i += 32) dst_p[dof + i] = i < cnt ? src_p[so + i] : 0.0f;
            }
        }
        if (src_l && dst_l && n_mels) {
            const uint64_t so = (uint64_t)f * n_mels, dof = (uint64_t)j * n_mels;
            if (vec_l) {
                const float4 *sp = reinterpret_cast<const float4 *>(src_l + so);
                float4 *dp = reinterpret_cast<float4 *>(dst_l + dof);
                for (uint32_t i = lane; i < n_mels / 4; i += 32) __stcs(dp + i, __ldcs(sp + i));
            } else {
                for (uint32_t i = lane; i < n_mels; i += 32) dst_l[dof + i] = src_l[so + i];
            }
        }
    }
}

cudaError_t launch_vad_gate(const GateJob &J, cudaStream_t st)
{
    if (J.n_streams == 0) return cudaSuccess;
    af_gate_offsets_kernel<<<J.n_streams, GATE_THREADS, 0, st>>>(J.seg, J.seg_cap, J.n_seg, J.off, J.total);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    if ((J.pcm && J.out_pcm) || (J.logmel && J.out_lm)) {
        const uint32_t gx = std::max<uint32_t>(1u, std::min<uint32_t>(1024u, (8u * 148u + J.n_streams - 1) / J.n_streams));
        af_gate_copy_kernel<<<dim3(gx, J.n_streams), GATE_THREADS, 0, st>>>(J.pcm, J.pcm_stride, J.logmel, J.logmel_stride, J.n_mels, J.n_out,
                                                                            J.hop, J.seg, J.seg_cap, J.n_seg, J.off, J.out_pcm,
                                                                            J.out_pcm_stride, J.out_lm, J.out_lm_stride);
        e = cudaGetLastError();
    }
    return e;
}

}  // namespace af
