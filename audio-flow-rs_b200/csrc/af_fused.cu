// af_fused.cu -- the fused hot-path kernel for sm_100a: one persistent CTA per SM, 28 warps in four
// roles that run concurrently on different steps (32 frames) of the CTA's tiles and hand buffers to
// each other through mbarriers -- there is no CTA-wide barrier after start-up.  Which hardware warp
// plays which role is a launch parameter (warp_role, af_common.cuh):
//
//   1 warp   "V"  issues the TMA bulk copies (cp.async.bulk + mbarrier complete_tx) that stage the raw
//                 interleaved input of each part of a step in shared memory from host-planned descriptors;
//                 then K4's energy part: one bit-exact 400-term sequential mean-square chain per lane (= frame)
//   7 warps  "R"  K1: downmix + cubic (rubato FastFixedIn) resample from the stage into the padded
//                 16 kHz step buffer (double buffered), PCM written to HBM straight from registers;
//                 publishes a StepInfo record per step for the roles downstream
//   16 warps "F"  K2: Hann window + 512-point real FFT (packed 256-point complex, 16 x 16 in registers in
//                 f32x2 arithmetic, one half-warp per frame, transposed through shared memory, Hermitian
//                 split by shuffles), power into pbuf[frame][bin]; per-lane constants from tensor memory
//   4 warps  "M"  K3: sparse banded mel projection + log, lane = frame, warp-uniform weight quads served
//                 from tensor memory (tcgen05.ld)
//
// Replaces capture.rs:30-42, resampler.rs:71-93/132-166 (+ rubato) and the O(len) part of
// vad.rs:157-168; the STFT/mel stages are spec-defined (DESIGN.md).  The sequential EMA/state
// machine of vad.rs:101-153 runs in the scan kernels (af_kernels.cu).
#include <atomic>
#include <type_traits>

// This file is compiled TWICE (Makefile).  The default translation unit holds the kernel all-48-kHz-mono-f32 batches run
// (cfg2): its resampler role is one loop over every kind of tile (role_resample_single).  With -DAF_FUSED_SPLIT_TU it
// holds the kernel of every other batch (cfg3, cfg4, sessions with other formats): the same roles, but the resampler role
// instantiates the steps of a tile twice -- 48 kHz mono f32 / everything else (role_resample_split).  Two units instead of
// one template parameter because the hot kernel is sensitive to what else is compiled next to it: as a third instance
// of one template it came out 3-7 % slower on cfg2 (0.585-0.595 vs 0.555 ms), in a unit of its own it is the kernel it was.
#ifdef AF_FUSED_SPLIT_TU
#define af_fused_kernel af_fused_split_kernel
#define g_pipe_stats g_pipe_stats_split
#endif

#include "af_device.cuh"
#include "af_launch.h"

namespace af {

constexpr int AF_MAX_GPUS_INTERNAL = 16;

// What the resampler warps need of a TileDev, copied as it lies in global memory: the 32-byte header and the 80 bytes
// behind the fill descriptors (stream descriptor + position increments).  cp.async puts the NEXT tile's copy into the
// warp's other slot while the current tile is worked on: no registers are held across the tile and nothing waits for
// the global loads (held in registers, the prefetched words were spilled at once -- a store that waits for the load).
struct alignas(16) RsTile {
    uint32_t stream_idx, tile;
    int tile_k;                                      // floor(position) of the tile's first output (TileDev::k0)
    uint32_t tile_rem;                               // and its remainder (numerator units)
    uint32_t n_steps, tile_end, n_frames, parts;
    StreamDev stream;
    uint32_t inc_k, inc_rem;                         // position increment for RS_THREADS outputs
};
static_assert(sizeof(RsTile) == 112 && offsetof(RsTile, stream) == 32, "RsTile mirrors the head and the tail of TileDev");
static_assert(offsetof(TileDev, sdesc) % 16 == 0 && sizeof(TileDev) - offsetof(TileDev, sdesc) == 80 && offsetof(TileDev, parts) == 28 &&
              offsetof(TileDev, inc_k) == offsetof(TileDev, sdesc) + sizeof(StreamDev), "TileDev layout the cp.async prefetch relies on");

struct __align__(128) FusedSmem {
    unsigned char stage[N_STAGE][STAGE_BYTES];       // raw interleaved input of a part of a step (bulk-copy targets)
    float ybuf[2][YBUF_FLOATS];                      // padded 16 kHz samples of two consecutive steps
    float scr[FFT_WARPS * SCR_FLOATS_PER_WARP];      // per FFT warp transpose scratch
    float pbuf[2][PBUF_FLOATS];                      // 4*|X[k]|^2, [pb_row(frame)][bin], two consecutive steps
    uint32_t tmem_base;                              // TMEM allocation holding the FFT constants (see tmem_* above)
    uint32_t pad_[3];
    StepInfo yinfo[2];                               // what ybuf[b] holds: written by resampler thread 0 before its y_full arrive
    StepInfo pinfo[4];                               // ring (step & 3) of what the power buffers hold: copied from yinfo by FFT
                                                     // thread 0 as soon as it sees a step, four deep so that no FFT lane has to
                                                     // carry the record across the transform (the mel warps lag < 3 steps)
    MelTables mel;
    // pipeline barriers (mbarriers): full = data ready for the consumer, empty = buffer may be overwritten
    unsigned long long stage_full[N_STAGE], stage_empty[N_STAGE];
    unsigned long long y_full[2], y_empty[2];
    unsigned long long p_full[2], p_empty[2];
    // metadata of the fill held by stage[h], written by the issuing thread before its arrive
    unsigned long long st_lo[N_STAGE], st_hi[N_STAGE];   // interleaved element range [lo, hi) held by the stage
    uint32_t st_interior[N_STAGE];                   // 1: every tap of the half step is inside the stage and the stream;
                                                     // 2: inside the stream but not staged (unchecked global loads)
    // resampler role: every warp keeps its own copy of the tile's stream descriptor and first-output position, so that
    // a new tile needs no synchronisation among the resampler warps
    RsTile rs[2][RS_WARPS];
    // periodic positions of the batch's table-mode rate (FusedParams::per_p / per_q): output r of a period of q outputs sits
    // floor((r + 1) p / q) input frames behind the period's base; sw_*: what a sweep of 4 * RS_THREADS outputs adds
    uint32_t per_p, per_q, sw_r, sw_kp;
    alignas(8) uint16_t koff[KOFF_MAX];
};
static_assert(sizeof(FusedSmem) <= 232448, "FusedSmem exceeds the 227 KB a CTA may use");

// ---- mbarrier / bulk-copy wrappers (PTX; SASS: SYNCS.*, UBLKCP) ----
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long *bar)
{
#ifdef AF_ARRIVE_RELAXED
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.relaxed.cta.shared::cta.b64 st, [%0];\n\t}" ::"r"(smem_u32(bar)) : "memory");
#else
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(smem_u32(bar)) : "memory");
#endif
}
__device__ __forceinline__ void mbar_arrive_expect_tx(unsigned long long *bar, uint32_t bytes)
{
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}" ::"r"(smem_u32(bar)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, uint32_t parity)
{
#ifdef AF_WAIT_SLEEP
    // poll with an explicit back-off: the "suspended" try_wait below comes back after a few cycles, so a waiting warp
    // spins at ~5 instructions + 2 barrier reads per 8 cycles (ncu: 50+ trips per wait) and takes issue slots and
    // shared-memory requests from the working warps
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "WAIT_%=:\n\t"
        "nanosleep.u32 %2;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@!p bra WAIT_%=;\n\t"
        "DONE_%=:\n\t"
        "}" ::"r"(smem_u32(bar)),
        "r"(parity), "n"(AF_WAIT_SLEEP)
        : "memory");
#else
    // try_wait with a suspend-time hint: the hardware parks the warp until the phase completes (or the hint
    // expires), so waiting warps do not take issue slots from the working ones
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
        "@!p bra WAIT_%=;\n\t"
        "}" ::"r"(smem_u32(bar)),
        "r"(parity), "r"(1000000u)
        : "memory");
#endif
}
// non-blocking phase test
__device__ __forceinline__ bool mbar_test(unsigned long long *bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0u;
}
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, unsigned long long *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void cp_async16(void *dst_smem, const void *src_gmem)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst_smem)), "l"(src_gmem) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
// warp-level arrive: every lane's earlier shared-memory accesses are ordered before lane 0's arrive
__device__ __forceinline__ void warp_arrive(unsigned long long *bar, int lane)
{
    __syncwarp();
    if (lane == 0) mbar_arrive(bar);
}
// global load the compiler cannot rematerialise at the use site: keeps per-lane constants in registers
__device__ __forceinline__ float2 ldg_f2_pinned(const void *p)
{
    float2 v;
    asm volatile("ld.global.nc.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "l"(p));
    return v;
}
__device__ __forceinline__ void named_bar_sync(int id, int count)
{
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory");
}
// optional pipeline statistics (make STATS=1): cycles each role spends in each of its waits, summed over warps
#ifdef AF_PIPE_STATS
__device__ unsigned long long g_pipe_stats[32];
#define AF_STATS_DECL long long ws_[7] = {0, 0, 0, 0, 0, 0, 0}; const long long ws_t0_ = clock64();
#define AF_WAIT(bar, parity, id) do { const long long t0_ = clock64(); mbar_wait(bar, parity); ws_[id] += clock64() - t0_; } while (0)
#define AF_TIC long long tic_ = clock64();
#define AF_TIC2 tic_ = clock64();
#define AF_TOC(id) ws_[id] += clock64() - tic_;
#define AF_STATS_FLUSH(role, lane) do { if ((lane) == 0) { atomicAdd(&g_pipe_stats[8 * (role)], (unsigned long long)(clock64() - ws_t0_)); \
    for (int i_ = 0; i_ < 7; ++i_) atomicAdd(&g_pipe_stats[8 * (role) + 1 + i_], (unsigned long long)ws_[i_]); } } while (0)
#else
#define AF_STATS_DECL
#define AF_TIC
#define AF_TIC2
#define AF_TOC(id)
#define AF_WAIT(bar, parity, id) mbar_wait(bar, parity)
#define AF_STATS_FLUSH(role, lane)
#endif


// ---- tensor memory (TMEM) as a per-lane constant store -------------------------------------------------------
// The FFT warps need 74 per-lane constants per frame pair (window samples, pass-1 and Hermitian-split twiddles).
// They do not fit the register budget, and as shared-memory loads they were 37 of ~236 LSU wavefronts per frame
// on an LSU-bound kernel.  TMEM is lane-addressed (thread t of a warp reads lane 32 (warp % 4) + t), has its own
// datapath (tcgen05.ld, no LSU / shared-memory bandwidth) and is otherwise idle here: the constants are written
// once per CTA into 74 columns of each lane quarter and fetched from there just before use.
constexpr uint32_t TM_TW1 = 0;               // 32 columns: tw1p[p] = columns 4p .. 4p+3  (re_a, re_b, im_a, im_b)
constexpr uint32_t TM_TW2 = 32;              // 16 columns: tw2p[r] = columns 4r .. 4r+3
constexpr uint32_t TM_WIN = 48;              // 26 columns: window[32 n1 + 2 l + e] at 2 n1 + e
__device__ __forceinline__ void tmem_alloc(uint32_t *smem_dst)
{
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr)
{
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(TMEM_COLS) : "memory");
}
__device__ __forceinline__ void tmem_st2(uint32_t taddr, float a, float b)
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1, %2};" ::"r"(taddr), "f"(a), "f"(b) : "memory");
}
__device__ __forceinline__ void tmem_st4(uint32_t taddr, float4 v)
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ float4 tmem_ld4(uint32_t taddr)
{
    float4 v;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(taddr));
    return v;
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float (&v)[8])
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]) : "r"(taddr));
}
__device__ __forceinline__ float2 tmem_ld2(uint32_t taddr)
{
    float2 v;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(taddr));
    return v;
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16])
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                 : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]), "=f"(v[8]),
                   "=f"(v[9]), "=f"(v[10]), "=f"(v[11]), "=f"(v[12]), "=f"(v[13]), "=f"(v[14]), "=f"(v[15])
                 : "r"(taddr));
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float4 &a, const float4 &b, const float4 &c, const float4 &d)
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
                 "f"(a.x), "f"(a.y), "f"(a.z), "f"(a.w), "f"(b.x), "f"(b.y), "f"(b.z), "f"(b.w), "f"(c.x), "f"(c.y), "f"(c.z), "f"(c.w),
                 "f"(d.x), "f"(d.y), "f"(d.z), "f"(d.w)
                 : "memory");
}
// the loaded registers may be used only after the wait: passing them through the statement as in/out operands
// keeps the compiler from scheduling a use above it
__device__ __forceinline__ void tmem_wait_ld(float4 &a)
{
    asm volatile("tcgen05.wait::ld.sync.aligned;" : "+f"(a.x), "+f"(a.y), "+f"(a.z), "+f"(a.w)::"memory");
}
__device__ __forceinline__ void tmem_wait_ld(float4 &a, float4 &b)
{
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+f"(a.x), "+f"(a.y), "+f"(a.z), "+f"(a.w), "+f"(b.x), "+f"(b.y), "+f"(b.z), "+f"(b.w)::"memory");
}
__device__ __forceinline__ void tmem_wait_ld(float (&v)[8])
{
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+f"(v[0]), "+f"(v[1]), "+f"(v[2]), "+f"(v[3]), "+f"(v[4]), "+f"(v[5]), "+f"(v[6]), "+f"(v[7])::"memory");
}
__device__ __forceinline__ void tmem_wait_ld(float (&v)[16])
{
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+f"(v[0]), "+f"(v[1]), "+f"(v[2]), "+f"(v[3]), "+f"(v[4]), "+f"(v[5]), "+f"(v[6]), "+f"(v[7]), "+f"(v[8]),
                   "+f"(v[9]), "+f"(v[10]), "+f"(v[11]), "+f"(v[12]), "+f"(v[13]), "+f"(v[14]), "+f"(v[15])::"memory");
}
__device__ __forceinline__ void tmem_wait_ld(float2 &a) { asm volatile("tcgen05.wait::ld.sync.aligned;" : "+f"(a.x), "+f"(a.y)::"memory"); }

// ---- geometry of a tile, recomputed by every role from the same tables ----
struct TileGeo {
    uint32_t stream, n_tile0, tile_end, f_tile0, n_steps, n_frames, parts;
};
__device__ __forceinline__ TileGeo tile_geo(const FusedParams &P, uint32_t tile, uint32_t *n_frames)
{
    const TileDev *td = P.tiles + tile;
    TileGeo t;
    t.stream = td->stream;
    t.n_tile0 = td->tile * TILE_SAMPLES;
    t.tile_end = td->tile_end;
    t.f_tile0 = td->tile * TILE_FRAMES;
    t.n_steps = td->n_steps;
    t.n_frames = td->n_frames;
    t.parts = td->parts;
    if (n_frames) *n_frames = td->n_frames;
    return t;
}
__device__ __forceinline__ int part_lo(uint32_t g, int parts, int k) { return k == 0 ? (g == 0 ? 0 : CARRY) : part_end(parts, k - 1); }

// ---- stage fill (descriptors planned per tile by plan_tile, af_device.cuh) ----
// issued by ONE thread; always completes one phase of stage_full[h]
__device__ __forceinline__ void issue_fill(FusedSmem &sm, const FusedParams &P, FillDesc d, int h)
{
    if (!P.use_stage) {                                  // "sync" variant: nothing staged
        d.bytes = 0; d.lo = 0; d.hi = 0;
        if (d.interior == 1u) d.interior = 2u;
    }
    sm.st_lo[h] = d.lo; sm.st_hi[h] = d.hi; sm.st_interior[h] = d.interior;
    if (d.bytes) {
        mbar_arrive_expect_tx(&sm.stage_full[h], d.bytes);
        bulk_g2s(sm.stage[h], d.src, d.bytes, &sm.stage_full[h]);
    } else {
        mbar_arrive(&sm.stage_full[h]);
    }
}

// ---- one mono input frame (downmixed) for the resampler, from the stage when it holds it ----
enum { K_F32_1 = 0, K_I16_1 = 1, K_F32_2 = 2, K_I16_2 = 3, K_GENERIC = 4 };

template <int KIND>
__device__ __forceinline__ float tap(const unsigned char *__restrict__ stage, const StreamDev &s, uint32_t st_lo,
                                     uint32_t st_hi, int idx)
{
    if ((uint32_t)idx >= s.n_in) return 0.0f;                        // also covers idx < 0
    if (KIND == K_F32_1) {
        const uint32_t e = (uint32_t)idx;
        if (e >= st_lo && e < st_hi) return reinterpret_cast<const float *>(stage)[e - st_lo];
        return __ldg(reinterpret_cast<const float *>(s.data) + e);
    } else if (KIND == K_I16_1) {
        const uint32_t e = (uint32_t)idx;
        short v;
        if (e >= st_lo && e < st_hi) v = reinterpret_cast<const short *>(stage)[e - st_lo];
        else v = __ldg(reinterpret_cast<const short *>(s.data) + e);
        return (float)v * (1.0f / 32768.0f);
    } else if (KIND == K_F32_2) {
        const uint32_t e = 2u * (uint32_t)idx;
        if (e >= st_lo && e + 2 <= st_hi) {
            const float2 v = *reinterpret_cast<const float2 *>(reinterpret_cast<const float *>(stage) + (e - st_lo));
            return __fmul_rn(__fadd_rn(__fadd_rn(0.0f, v.x), v.y), 0.5f);
        }
        return load_mono(s.data, s.n_samples, s.n_in, 2, FMT_F32, idx);
    } else if (KIND == K_I16_2) {
        const uint32_t e = 2u * (uint32_t)idx;
        if (e >= st_lo && e + 2 <= st_hi) {
            const short2 v = *reinterpret_cast<const short2 *>(reinterpret_cast<const short *>(stage) + (e - st_lo));
            const float l = (float)v.x * (1.0f / 32768.0f), r = (float)v.y * (1.0f / 32768.0f);
            return __fmul_rn(__fadd_rn(__fadd_rn(0.0f, l), r), 0.5f);
        }
        return load_mono(s.data, s.n_samples, s.n_in, 2, FMT_I16, idx);
    } else {
        return load_mono(s.data, s.n_samples, s.n_in, s.channels, s.format, idx);
    }
}

// unchecked tap for interior steps: `off` = mono frame index relative to the first staged frame
template <int KIND>
__device__ __forceinline__ float tap_fast(const unsigned char *stage, int off)
{
    if (KIND == K_F32_1) return reinterpret_cast<const float *>(stage)[off];
    if (KIND == K_I16_1) return (float)reinterpret_cast<const short *>(stage)[off] * (1.0f / 32768.0f);
    if (KIND == K_F32_2) {
        const float2 v = reinterpret_cast<const float2 *>(stage)[off];
        return __fmul_rn(__fadd_rn(__fadd_rn(0.0f, v.x), v.y), 0.5f);
    }
    const short2 v = reinterpret_cast<const short2 *>(stage)[off];
    const float l = (float)v.x * (1.0f / 32768.0f), r = (float)v.y * (1.0f / 32768.0f);
    return __fmul_rn(__fadd_rn(__fadd_rn(0.0f, l), r), 0.5f);
}

// one resampled sample leaves its producer twice: into the step buffer and (its owner tile only) to HBM
struct YSink {
    float *__restrict__ yb;       // step buffer
    float *__restrict__ pcm;      // stream's PCM row or nullptr
    uint32_t base;                // stream index of step-buffer sample 0
    uint32_t wr_end;              // the tile owns stream samples < wr_end
    float nz;                     // FusedParams::neg_zero (interp_cubic2)
    __device__ __forceinline__ void put(int i, float v) const
    {
        yb[ypad(i)] = v;
        const uint32_t n = base + (uint32_t)i;
        if (pcm && n < wr_end) __stcs(pcm + n, v);
    }
    __device__ __forceinline__ void put4(int i4, float4 y) const
    {
        *reinterpret_cast<float4 *>(yb + ypad(i4)) = y;
        const uint32_t n = base + (uint32_t)i4;
        if (pcm) {
            if (n + 4 <= wr_end) __stcs(reinterpret_cast<float4 *>(pcm + n), y);
            else {
                if (n < wr_end) __stcs(pcm + n, y.x);
                if (n + 1 < wr_end) __stcs(pcm + n + 1, y.y);
                if (n + 2 < wr_end) __stcs(pcm + n + 2, y.z);
            }
        }
    }
};

// ---- the hot resampling loop: 48 kHz -> 16 kHz mono f32, interior half step, taps in the stage ----
// x0 points at the tap y0 of step-buffer sample 0 (output n reads x0[3n .. 3n+3]); outputs [i_lo, i_hi) of the step go
// to yb (padded) and to pq0[i] (the PCM row, nullptr-based offsets never dereferenced when lim4 is the "no PCM" value).
__device__ __forceinline__ void resample_quads_48k(const float *__restrict__ x0, float *__restrict__ yb, float *pq0, int lim4,
                                                   int i_lo, int i_hi, int rtid)
{
        constexpr int QS = 4 * RS_THREADS;                       // outputs per sweep of the resampler warps (7 x 32 quads)
        static_assert(QS % 32 == 0, "a sweep must keep the 32-sample padding phase");
        int i4 = (i_lo & ~31) + 4 * rtid;
        if (i4 < i_lo) i4 += QS;
        const float *px = x0 + 3 * i4;
        float *yq = yb + ypad(i4);
        float *pq = pq0 + i4;
        auto quad = [&](const float *p, float *ydst, float *pdst, int i) {
            const float2 hh = *reinterpret_cast<const float2 *>(p);
            const float4 a4 = *reinterpret_cast<const float4 *>(p + 2);
            const float4 b4 = *reinterpret_cast<const float4 *>(p + 6);
            const float4 c4 = *reinterpret_cast<const float4 *>(p + 10);
            // frac == 0: the cubic returns y1 bit for bit when y1 != 0 and every tap is finite with |x| < 2 (exponent
            // bit 30 clear in the OR of the 13 words: covers Inf / NaN); anything else takes the polynomial
            const uint32_t orx = (__float_as_uint(hh.x) | __float_as_uint(hh.y) | __float_as_uint(a4.x)) |
                                 (__float_as_uint(a4.y) | __float_as_uint(a4.z) | __float_as_uint(a4.w)) |
                                 (__float_as_uint(b4.x) | __float_as_uint(b4.y) | __float_as_uint(b4.z)) |
                                 (__float_as_uint(b4.w) | __float_as_uint(c4.x) | __float_as_uint(c4.y)) | __float_as_uint(c4.z);
            float4 y = make_float4(hh.y, a4.z, b4.y, c4.x);
            if (!((orx & 0x40000000u) == 0u && y.x != 0.0f && y.y != 0.0f && y.z != 0.0f && y.w != 0.0f)) {
                y.x = interp_cubic(0.0f, hh.x, hh.y, a4.x, a4.y);
                y.y = interp_cubic(0.0f, a4.y, a4.z, a4.w, b4.x);
                y.z = interp_cubic(0.0f, b4.x, b4.y, b4.z, b4.w);
                y.w = interp_cubic(0.0f, b4.w, c4.x, c4.y, c4.z);
            }
            *reinterpret_cast<float4 *>(ydst) = y;
            if (i <= lim4) __stcs(reinterpret_cast<float4 *>(pdst), y);
            else {                                                // the quad straddles (or lies beyond) the end of the owner tile
                const int left = lim4 + 4 - i;
                if (left > 0) __stcs(pdst, y.x);
                if (left > 1) __stcs(pdst + 1, y.y);
                if (left > 2) __stcs(pdst + 2, y.z);
            }
        };
        for (; i4 + QS < i_hi; i4 += 2 * QS) {
            quad(px, yq, pq, i4);
            quad(px + 3 * QS, yq + ypad(QS), pq + QS, i4 + QS);
            px += 6 * QS; yq += 2 * ypad(QS); pq += 2 * QS;
        }
        if (i4 < i_hi) quad(px, yq, pq, i4);
}

// ---- the same for 48 kHz STEREO f32 (cfg4): four outputs per thread and quad from 14 stereo frames = seven LDS.128 ----
// x0 points at the stereo frame of tap y0 of step-buffer sample 0.  For a quad (i4 = 0 mod 4) the first frame it reads,
// 3 i4 - 1 past x0's frame, is even relative to a 16-byte boundary of the stage, so the 28 floats are seven aligned float4.
// Downmix as AudioFrame::to_mono does ((0 + l) + r) / 2, in packed arithmetic (an addition followed by a multiplication:
// nothing ptxas could contract), then the mono quad's test for the bit-exact frac = 0 shortcut.
__device__ __forceinline__ void resample_quads_48k_stereo(const float *__restrict__ x0, float *__restrict__ yb, float *pq0, int lim4,
                                                          int i_lo, int i_hi, int rtid)
{
    constexpr int QS = 4 * RS_THREADS;
    int i4 = (i_lo & ~31) + 4 * rtid;
    if (i4 < i_lo) i4 += QS;
    const float4 *px = reinterpret_cast<const float4 *>(x0 + 6 * i4);          // 3 frames x 2 floats per output
    float *yq = yb + ypad(i4);
    float *pq = pq0 + i4;
    const f2 zero = mk2(0.0f, 0.0f), half = mk2(0.5f, 0.5f);
    for (; i4 < i_hi; i4 += QS) {
        float m[14];                                                            // mono frames 3 i4 - 1 ... 3 i4 + 12 (the last is not used)
#pragma unroll
        for (int j = 0; j < 7; ++j) {
            const float4 v = px[j];                                             // frames 2 j, 2 j + 1 of the quad: (l, r, l, r)
            const f2 mm = mul2(add2(add2(zero, mk2(v.x, v.z)), mk2(v.y, v.w)), half);
            m[2 * j] = mm.x; m[2 * j + 1] = mm.y;
        }
        uint32_t orx = 0;
#pragma unroll
        for (int j = 0; j < 13; ++j) orx |= __float_as_uint(m[j]);
        float4 y = make_float4(m[1], m[4], m[7], m[10]);
        if (!((orx & 0x40000000u) == 0u && y.x != 0.0f && y.y != 0.0f && y.z != 0.0f && y.w != 0.0f)) {
            y.x = interp_cubic(0.0f, m[0], m[1], m[2], m[3]);
            y.y = interp_cubic(0.0f, m[3], m[4], m[5], m[6]);
            y.z = interp_cubic(0.0f, m[6], m[7], m[8], m[9]);
            y.w = interp_cubic(0.0f, m[9], m[10], m[11], m[12]);
        }
        *reinterpret_cast<float4 *>(yq) = y;
        if (i4 <= lim4) __stcs(reinterpret_cast<float4 *>(pq), y);
        else {
            const int left = lim4 + 4 - i4;
            if (left > 0) __stcs(pq, y.x);
            if (left > 1) __stcs(pq + 1, y.y);
            if (left > 2) __stcs(pq + 2, y.z);
        }
        px += 6 * QS / 4; yq += ypad(QS); pq += QS;
    }
}

// ---- general rational step, interior part (44.1 kHz -> 16 kHz: 441/160 with table fractions; 8 / 24 / 32 kHz: exact) ----
// Four consecutive outputs per thread and quad: exact integer positions advanced by p / q per output, 16 unchecked taps,
// four unfused cubics (the reference's operation order), one 16-byte store to the step buffer and one to HBM.  The table
// fractions of a quad (one 16-byte load from L2) are requested one quad AHEAD, so that the round trip overlaps the
// arithmetic of the quad before it; their sign bit says "one tap earlier" (plan_rate), which saves the float round trip
// the position correction used to take.  srcp: the stage (first staged mono frame f_lo) or the stream itself (f_lo = 0).
template <int KIND>
__device__ __forceinline__ void resample_part_rational(const unsigned char *__restrict__ srcp, int tile_k, uint32_t tile_rem,
                                                       const StreamDev *__restrict__ sp, const YSink &out, uint32_t tile_off, int i_lo,
                                                       int i_hi, int rtid, int f_lo, float nz)
{
    constexpr int QS = 4 * RS_THREADS;
    const uint32_t p = sp->p, q = sp->q;
    const bool table = sp->mode == RS_TABLE;
    int i4 = (i_lo & ~31) + 4 * rtid;
    if (i4 < i_lo) i4 += QS;
    if (i4 >= i_hi) return;
    const float4 *__restrict__ frac4 = reinterpret_cast<const float4 *>(sp->frac + out.base + i4);
    float4 ft = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    if (table) ft = __ldg(frac4);
    const uint32_t a0 = tile_rem + (tile_off + (uint32_t)i4) * p;
    uint32_t dk = a0 / q, rem = a0 - dk * q;
    int k = tile_k + (int)dk - 1 - f_lo;                     // tap y0 of output i4, relative to the staged frames
    const uint32_t pk = p / q, pr = p - pk * q;              // per output
    const uint32_t sweep = (uint32_t)(QS - 3) * p;           // from the quad's last output to the next sweep's first
    const uint32_t sk = sweep / q, sr = sweep - sk * q;
    const float inv_q = 1.0f / (float)q;
    const int lim4 = out.pcm ? (int)min((uint32_t)YLEN, out.wr_end - min(out.wr_end, out.base)) - 4 : -(1 << 30);
    float *yq = out.yb + ypad(i4);
    float *pq = out.pcm + out.base + i4;
    for (; i4 < i_hi; i4 += QS) {
        frac4 += QS / 4;
        float4 ft_next = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        if (table && i4 + QS < i_hi) ft_next = __ldg(frac4);
        const float fq[4] = {ft.x, ft.y, ft.z, ft.w};
        float fr[4], t0[4], t1[4], t2[4], t3[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            int o = k;
            if (table) { o -= (int)(__float_as_uint(fq[u]) >> 31); fr[u] = fabsf(fq[u]); }
            else fr[u] = (float)rem * inv_q;                 // RS_EXACT: q is a power of two, exact
            t0[u] = tap_fast<KIND>(srcp, o); t1[u] = tap_fast<KIND>(srcp, o + 1);
            t2[u] = tap_fast<KIND>(srcp, o + 2); t3[u] = tap_fast<KIND>(srcp, o + 3);
            if (u < 3) {
                k += (int)pk; rem += pr;
                if (rem >= q) { rem -= q; k += 1; }
            }
        }
        // two outputs per packed cubic (bit for bit the scalar interp_cubic: see interp_cubic2)
        const f2 ya = interp_cubic2(mk2(fr[0], fr[1]), mk2(t0[0], t0[1]), mk2(t1[0], t1[1]), mk2(t2[0], t2[1]), mk2(t3[0], t3[1]), nz);
        const f2 yb2 = interp_cubic2(mk2(fr[2], fr[3]), mk2(t0[2], t0[3]), mk2(t1[2], t1[3]), mk2(t2[2], t2[3]), mk2(t3[2], t3[3]), nz);
        const float4 yv = make_float4(ya.x, ya.y, yb2.x, yb2.y);
        *reinterpret_cast<float4 *>(yq) = yv;
        if (i4 <= lim4) __stcs(reinterpret_cast<float4 *>(pq), yv);
        else {
            const int left = lim4 + 4 - i4;
            if (left > 0) __stcs(pq, yv.x);
            if (left > 1) __stcs(pq + 1, yv.y);
            if (left > 2) __stcs(pq + 2, yv.z);
        }
        k += (int)sk; rem += sr;
        if (rem >= q) { rem -= q; k += 1; }
        yq += ypad(QS); pq += QS;
        ft = ft_next;
    }
}

// ---- table-mode rate whose positions repeat every q outputs (44.1 kHz -> 16 kHz: q = 160, p = 441), interior part ----
// Output i of the step buffer (the step starts on a period boundary: q divides STEP_SAMPLES) reads the taps
// kb + (i div q) p + koff[i mod q] - 1 ...: one LDS.64 of four 16-bit offsets replaces the quad's position arithmetic, the
// period counter advances by constants per sweep.  Fractions as in resample_part_rational (table in L2, one quad ahead).
template <int KIND>
__device__ __forceinline__ void resample_part_periodic(const FusedSmem &sm, const unsigned char *__restrict__ srcp, int kb, uint32_t p,
                                                       uint32_t q, const float *__restrict__ frac_row, const YSink &out, int i_lo, int i_hi,
                                                       int rtid)
{
    constexpr int QS = 4 * RS_THREADS;
    int i4 = (i_lo & ~31) + 4 * rtid;
    if (i4 < i_lo) i4 += QS;
    if (i4 >= i_hi) return;
    const float4 *__restrict__ frac4 = reinterpret_cast<const float4 *>(frac_row + i4);
    float4 ft = __ldg(frac4);
    const uint32_t per = (uint32_t)i4 / q;
    uint32_t r4 = (uint32_t)i4 - per * q;                    // position of the quad inside its period (a multiple of 4)
    kb += (int)(per * p);
    const uint32_t sw_r = sm.sw_r;
    const int sw_kp = (int)sm.sw_kp;
    const int lim4 = out.pcm ? (int)min((uint32_t)YLEN, out.wr_end - min(out.wr_end, out.base)) - 4 : -(1 << 30);
    float *yq = out.yb + ypad(i4);
    float *pq = out.pcm + out.base + i4;
    for (; i4 < i_hi; i4 += QS) {
        frac4 += QS / 4;
        float4 ft_next = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        if (i4 + QS < i_hi) ft_next = __ldg(frac4);
        const uint2 kk = *reinterpret_cast<const uint2 *>(sm.koff + r4);
        const uint32_t fb[4] = {__float_as_uint(ft.x), __float_as_uint(ft.y), __float_as_uint(ft.z), __float_as_uint(ft.w)};
        const uint32_t ko[4] = {kk.x & 0xffffu, kk.x >> 16, kk.y & 0xffffu, kk.y >> 16};
        float fr[4], t0[4], t1[4], t2[4], t3[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int o = kb + (int)ko[u] - (int)(fb[u] >> 31);      // sign bit: "one tap earlier" (plan_rate)
            fr[u] = __uint_as_float(fb[u] & 0x7fffffffu);
            t0[u] = tap_fast<KIND>(srcp, o); t1[u] = tap_fast<KIND>(srcp, o + 1);
            t2[u] = tap_fast<KIND>(srcp, o + 2); t3[u] = tap_fast<KIND>(srcp, o + 3);
        }
        const f2 ya = interp_cubic2(mk2(fr[0], fr[1]), mk2(t0[0], t0[1]), mk2(t1[0], t1[1]), mk2(t2[0], t2[1]), mk2(t3[0], t3[1]), out.nz);
        const f2 yb2 = interp_cubic2(mk2(fr[2], fr[3]), mk2(t0[2], t0[3]), mk2(t1[2], t1[3]), mk2(t2[2], t2[3]), mk2(t3[2], t3[3]), out.nz);
        const float4 yv = make_float4(ya.x, ya.y, yb2.x, yb2.y);
        *reinterpret_cast<float4 *>(yq) = yv;
        if (i4 <= lim4) __stcs(reinterpret_cast<float4 *>(pq), yv);
        else {
            const int left = lim4 + 4 - i4;
            if (left > 0) __stcs(pq, yv.x);
            if (left > 1) __stcs(pq + 1, yv.y);
            if (left > 2) __stcs(pq + 2, yv.z);
        }
        r4 += sw_r; kb += sw_kp;
        if (r4 >= q) { r4 -= q; kb += (int)p; }
        yq += ypad(QS); pq += QS;
        ft = ft_next;
    }
}

// ---- resampling, interior half steps: every tap comes unchecked from the stage (or the stream) ----
template <int KIND, bool STAGED>
__device__ __forceinline__ void resample_half_fast(const FusedSmem &sm, const RsTile &rt, int h, const StreamDev &s, const YSink &out,
                                                   uint32_t tile_off, int i_lo, int i_hi, int rtid)
{
    // taps come from the shared-memory stage (first staged mono frame f_lo) or, when the half step does not fit the
    // stage (e.g. stereo f32), unchecked from the stream in global memory (f_lo = 0)
    const unsigned char *__restrict__ srcp = STAGED ? sm.stage[h] : reinterpret_cast<const unsigned char *>(s.data);
    const int f_lo = STAGED ? (int)((uint32_t)sm.st_lo[h] / ((KIND == K_F32_2 || KIND == K_I16_2) ? 2u : 1u)) : 0;
    const uint32_t mode = s.mode;
    int i = i_lo + rtid;
    if (mode == RS_PASSTHROUGH) {
        for (; i < i_hi; i += RS_THREADS) out.put(i, tap_fast<KIND>(srcp, (int)(out.base + i) - f_lo));
        return;
    }
    const uint32_t q = s.q;
    if (KIND == K_F32_1 && q == 1 && s.p == 3) {
        // 48 kHz -> 16 kHz mono f32, four outputs per thread and quad: output n reads x[3n-2 .. 3n+1]; for n = 0 mod 4
        // that is an 8-byte aligned float2 followed by three 16-byte aligned float4 of the stage (14 floats, 13 used).
        // Two quads per iteration (independent instruction streams), all pointers advanced by constants.
        // Quads start on a 32-sample boundary of the padded step buffer: every quarter-warp stores 128 contiguous bytes.
        const int lim4 = out.pcm ? (int)min((uint32_t)YLEN, out.wr_end - min(out.wr_end, out.base)) - 4 : -(1 << 30);
        resample_quads_48k(reinterpret_cast<const float *>(srcp) + (rt.tile_k + 3 * (int)tile_off - 1 - f_lo), out.yb,
                           out.pcm + out.base, lim4, i_lo, i_hi, rtid);
        return;
    }
    const uint32_t a = rt.tile_rem + (tile_off + (uint32_t)i) * s.p;
    // An integer ratio whose f64 step is not exactly p (784 kHz, 1.488 MHz) is a TABLE rate with q == 1: its fractions are
    // not zero and may flag the tap below, so it takes resample_part_rational.  Only the split unit meets such streams (the
    // default one runs 48 kHz mono f32 alone), and the hot kernel keeps the code it had without the test.
#ifdef AF_FUSED_SPLIT_TU
    constexpr bool TABLE_Q1 = true;
#else
    constexpr bool TABLE_Q1 = false;
#endif
    if (q == 1 && (!TABLE_Q1 || mode == RS_EXACT)) {
        // integer step (48 kHz -> 16 kHz): frac == 0 exactly; the cubic returns y1 bit for bit whenever y1 != 0 and
        // the taps are finite with |x| < 2 -- checked per sample, everything else takes the polynomial
        int o = rt.tile_k + (int)a - 1 - f_lo;
        const int inc = (int)rt.inc_k;
#pragma unroll 2
        for (; i < i_hi; i += RS_THREADS, o += inc) {
            const float y0 = tap_fast<KIND>(srcp, o), y1 = tap_fast<KIND>(srcp, o + 1);
            const float y2 = tap_fast<KIND>(srcp, o + 2), y3 = tap_fast<KIND>(srcp, o + 3);
            const uint32_t orx = __float_as_uint(y0) | __float_as_uint(y1) | __float_as_uint(y2) | __float_as_uint(y3);
            float v = y1;
            if (!(y1 != 0.0f && (orx & 0x40000000u) == 0u)) v = interp_cubic(0.0f, y0, y1, y2, y3);
            out.put(i, v);
        }
        return;
    }
    if (s.mode == RS_TABLE && q == sm.per_q && s.p == sm.per_p) {
        // k of step-buffer output i = kb0 + (i div q) p + koff[i mod q]; tile_k is the k of the tile's first output (koff[0] past its
        // period base), the step starts tile_off / q periods later; "- 1 - f_lo": tap y0, relative to the staged frames
        const int kb0 = rt.tile_k - (int)sm.koff[0] + (int)((tile_off / q) * s.p) - 1 - f_lo;
        resample_part_periodic<KIND>(sm, srcp, kb0, s.p, q, s.frac + out.base, out, i_lo, i_hi, rtid);
        return;
    }
    resample_part_rational<KIND>(srcp, rt.tile_k, rt.tile_rem, &s, out, tile_off, i_lo, i_hi, rtid, f_lo, out.nz);
}

// ---- resampling, checked: samples [base + i_lo, base + i_hi) of the stream, zero beyond n_out ----
template <int KIND>
__device__ __noinline__ void resample_half(const FusedSmem &sm, const RsTile &rt, int h, const StreamDev &s, const YSink out,
                                           uint32_t tile_off, int i_lo, int i_hi, int rtid)
{
    const unsigned char *__restrict__ stage = sm.stage[h];
    const uint32_t st_lo = (uint32_t)sm.st_lo[h], st_hi = (uint32_t)sm.st_hi[h];
    const uint32_t n_out = s.n_out, mode = s.mode;
    int i = i_lo + rtid;
    if (mode == RS_PASSTHROUGH) {
        for (; i < i_hi; i += RS_THREADS) {
            const uint32_t n = out.base + i;
            out.put(i, n < n_out ? tap<KIND>(stage, s, st_lo, st_hi, (int)n) : 0.0f);
        }
        return;
    }
    // exact integer position of this thread's first output, relative to the tile start
    const uint32_t q = s.q;
    const uint32_t a = rt.tile_rem + (tile_off + (uint32_t)i) * s.p;
    uint32_t dk, rem;
    if (q == 1) { dk = a; rem = 0; }
    else { dk = a / q; rem = a - dk * q; }
    int k = rt.tile_k + (int)dk;
    const uint32_t inc_k = rt.inc_k, inc_rem = rt.inc_rem;
    const float inv_q = 1.0f / (float)q;
    const float *__restrict__ frac_tab = s.frac;
    for (; i < i_hi; i += RS_THREADS) {
        const uint32_t n = out.base + i;
        float v = 0.0f;
        if (n < n_out) {
            int kk = k;
            float frac;
            if (mode == RS_TABLE) {
                const float fe = __ldg(frac_tab + n);                 // sign bit: the f64 recurrence sits just below an integer (plan_rate)
                kk -= (int)(__float_as_uint(fe) >> 31);
                frac = fabsf(fe);
            } else {
                frac = (float)rem * inv_q;                            // q is a power of two: exact
            }
            const float y0 = tap<KIND>(stage, s, st_lo, st_hi, kk - 1);
            const float y1 = tap<KIND>(stage, s, st_lo, st_hi, kk);
            const float y2 = tap<KIND>(stage, s, st_lo, st_hi, kk + 1);
            const float y3 = tap<KIND>(stage, s, st_lo, st_hi, kk + 2);
            // frac == 0 (48 kHz -> 16 kHz): a0 + a1*0 + a2*0 + a3*0 == y1 bit for bit whenever y1 != 0 and the
            // coefficients are finite; only then skip the polynomial
            const uint32_t orx = __float_as_uint(y0) | __float_as_uint(y1) | __float_as_uint(y2) | __float_as_uint(y3);
            if (frac == 0.0f && y1 != 0.0f && (orx & 0x40000000u) == 0u) v = y1;
            else v = interp_cubic(frac, y0, y1, y2, y3);
        }
        out.put(i, v);
        k += (int)inc_k;
        rem += inc_rem;
        if (rem >= q) { rem -= q; k += 1; }
    }
}

template <int KIND>
__device__ __forceinline__ void resample_dispatch(const FusedSmem &sm, const RsTile &rt, int h, const StreamDev &s, const YSink &out,
                                                  uint32_t tile_off, int i_lo, int i_hi, int rtid)
{
    const uint32_t interior = sm.st_interior[h];
    if (KIND != K_GENERIC && interior == 1) resample_half_fast<KIND, true>(sm, rt, h, s, out, tile_off, i_lo, i_hi, rtid);
    else if (KIND != K_GENERIC && interior == 2) resample_half_fast<KIND, false>(sm, rt, h, s, out, tile_off, i_lo, i_hi, rtid);
    else resample_half<KIND>(sm, rt, h, s, out, tile_off, i_lo, i_hi, rtid);
}

// ---- F role: one frame per half-warp, packed (f32x2) arithmetic: pack k = points 2k, 2k+1 of the lane ----
// window + pack: this lane holds z[16 n1 + l] = x[32 n1 + 2 l] + i x[32 n1 + 2 l + 1] of frame q as point n1
__device__ __forceinline__ void fft_load(const float *__restrict__ ybuf, uint32_t tm, int q, int l, f2 (&R)[8], f2 (&I)[8])
{
    const float *yb = ybuf + 180 * q + 2 * l;      // ypad(160 q + 32 n1 + 2 l) = 180 q + 36 n1 + 2 l
    // window samples of this lane from TMEM, in three batches so that few registers are held at a time
    float w[8];
#pragma unroll
    for (int g = 0; g < 3; ++g) {
        tmem_ld8(tm + TM_WIN + 8 * g, w);
        float2 v[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = *reinterpret_cast<const float2 *>(yb + 36 * (4 * g + j));
        tmem_wait_ld(w);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int n1 = 4 * g + j;
            const float re = __fmul_rn(v[j].x, w[2 * j]), im = __fmul_rn(v[j].y, w[2 * j + 1]);
            if (n1 & 1) { R[n1 >> 1].y = re; I[n1 >> 1].y = im; }
            else { R[n1 >> 1].x = re; I[n1 >> 1].x = im; }
        }
    }
    {
        float2 wl = tmem_ld2(tm + TM_WIN + 24);
        float2 v = make_float2(0.0f, 0.0f);
        if (l < 8) v = *reinterpret_cast<const float2 *>(yb + 36 * 12);   // samples 384 + 2l (+1) < 400; the window is 0 beyond
        tmem_wait_ld(wl);
        R[6] = mk2(__fmul_rn(v.x, wl.x), 0.0f);
        I[6] = mk2(__fmul_rn(v.y, wl.y), 0.0f);
    }
    R[7] = mk2(0.0f, 0.0f); I[7] = mk2(0.0f, 0.0f);
}

// the two 16-point passes of the packed 256-point transform; leaves Z[l + 16 k2] in slot(k2).  The 16 x 16
// transpose between them goes through the warp's scratch twice, real parts first, then imaginary parts.
__device__ __forceinline__ float &slot_of(f2 (&A)[8], int s) { return (s & 1) ? A[s >> 1].y : A[s >> 1].x; }
__device__ __forceinline__ void fft_passes(uint32_t tm, float *__restrict__ scr, int l, f2 (&R)[8], f2 (&I)[8])
{
    // pass 1: 16-point FFT over n1 (this lane is n2 = l), twiddle W256^(l k1) on the packs
    fft16p<true>(R, I);
#pragma unroll
    for (int g = 0; g < 4; ++g) {                   // two packs per TMEM round trip
        float4 wa = tmem_ld4(tm + TM_TW1 + 8 * g), wb = tmem_ld4(tm + TM_TW1 + 8 * g + 4);
        tmem_wait_ld(wa, wb);
        cmul2(R[2 * g], I[2 * g], mk2(wa.x, wa.y), mk2(wa.z, wa.w));
        cmul2(R[2 * g + 1], I[2 * g + 1], mk2(wb.x, wb.y), mk2(wb.z, wb.w));
    }
    // transposed store / load: this lane becomes k1 = l and reads its row (all n2)
#pragma unroll
    for (int k1 = 0; k1 < 16; ++k1) scr[k1 * SCR_ROW + l] = slot_of(R, fft16_slot(k1));
    __syncwarp();
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        const float4 v = *reinterpret_cast<const float4 *>(scr + l * SCR_ROW + 4 * u);
        R[2 * u] = mk2(v.x, v.y); R[2 * u + 1] = mk2(v.z, v.w);
    }
    __syncwarp();
#pragma unroll
    for (int k1 = 0; k1 < 16; ++k1) scr[k1 * SCR_ROW + l] = slot_of(I, fft16_slot(k1));
    __syncwarp();
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        const float4 v = *reinterpret_cast<const float4 *>(scr + l * SCR_ROW + 4 * u);
        I[2 * u] = mk2(v.x, v.y); I[2 * u + 1] = mk2(v.z, v.w);
    }
    __syncwarp();
    // pass 2: 16-point FFT over n2
    fft16p<false>(R, I);
}

// Hermitian split + power -> row pb_row(q) of pbuf, two bins r and r + 4 per pack.  Z[l + 16 k2] is in slot(k2) =
// 4 (k2 & 3) + (k2 >> 2): k2 = r and r + 4 are the two halves of pack 2 r.  Bin k = l + 16 k2 pairs with 256 - k,
// which lives in lane (16 - l) & 15 at k2' = 15 - k2 (lane 0 pairs with itself at k2' = (16 - k2) & 15).
__device__ __forceinline__ void fft_power(float *__restrict__ pbuf, uint32_t tm, int q, int l, int lane,
                                          f2 (&R)[8], f2 (&I)[8])
{
    const int src = ((16 - l) & 15) | (lane & 16);
    float *pb = pbuf + pb_row(q) * PB_ROW;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const f2 zr = R[2 * r], zi = I[2 * r];                           // k2 = r (x), r + 4 (y)
        // partners k2' = 15 - r -> slot 4 (3 - r) + 3 = pack 7 - 2 r half y;  k2' = 11 - r -> slot 4 (3 - r) + 2 = same pack half x
        f2 pr, pi;
        pr.x = __shfl_sync(0xffffffffu, R[7 - 2 * r].y, src); pi.x = __shfl_sync(0xffffffffu, I[7 - 2 * r].y, src);
        pr.y = __shfl_sync(0xffffffffu, R[7 - 2 * r].x, src); pi.y = __shfl_sync(0xffffffffu, I[7 - 2 * r].x, src);
        if (l == 0) {                                                    // own values at k2' = (16 - k2) & 15
            pr.x = slot_of(R, fft16_slot((16 - r) & 15)); pi.x = slot_of(I, fft16_slot((16 - r) & 15));
            pr.y = slot_of(R, fft16_slot(12 - r));        pi.y = slot_of(I, fft16_slot(12 - r));
        }
        float4 w = tmem_ld4(tm + TM_TW2 + 4 * r);
        tmem_wait_ld(w);
        const f2 wx = mk2(w.x, w.y), wy = mk2(w.z, w.w);
        const f2 e2r = add2(zr, pr), e2i = sub2(zi, pi);                 // 2E = Z[k] + conj(Z[256-k])
        const f2 o2r = add2(zi, pi), o2i = sub2(pr, zr);                 // 2O = -i (Z[k] - conj(Z[256-k]))
        const f2 tr = fma2(mk2(-wy.x, -wy.y), o2i, mul2(wx, o2r));
        const f2 ti = fma2(wy, o2r, mul2(wx, o2i));
        const f2 ar = add2(e2r, tr), ai = add2(e2i, ti);                 // 2 X[k]
        const f2 br = sub2(e2r, tr), bi = sub2(e2i, ti);                 // 2 conj(X[256-k])
        const f2 pa = fma2(ai, ai, mul2(ar, ar)), pbv = fma2(bi, bi, mul2(br, br));
        const int k = l + 16 * r;
        pb[k] = pa.x; pb[k + 64] = pa.y;
        pb[256 - k] = pbv.x; pb[192 - k] = pbv.y;
    }
    if (l == 0) {                                       // k = 128 (k2 = 8) pairs with itself
        const float zr = slot_of(R, fft16_slot(8)), zi = slot_of(I, fft16_slot(8));
        pb[128] = 4.0f * (zr * zr + zi * zi);
    }
}

// ---- V role, lane = frame: calculate_energy (vad.rs:157-168), strictly sequential ----
// The squares are independent (packed multiplies, two per instruction); the additions are one dependent chain in
// the reference's order.  `between()` runs after every 128 samples: the V warp's opportunistic fill service.
__device__ __forceinline__ float energy_acc4(float sum, float4 v)
{
    const f2 a = mul2(mk2(v.x, v.y), mk2(v.x, v.y)), b = mul2(mk2(v.z, v.w), mk2(v.z, v.w));
    sum = __fadd_rn(sum, a.x); sum = __fadd_rn(sum, a.y);
    sum = __fadd_rn(sum, b.x); sum = __fadd_rn(sum, b.y);
    return sum;
}
template <class F>
__device__ __forceinline__ float frame_energy_smem(const float *__restrict__ ybuf, int q, F between)
{
    const float4 *yp = reinterpret_cast<const float4 *>(ybuf) + 45 * q;   // ypad(160 q) / 4
    float sum = 0.0f;
#pragma unroll 1
    for (int seg = 0; seg < 3; ++seg) {
#pragma unroll 2
        for (int s8 = 4 * seg; s8 < 4 * seg + 4; ++s8) {
#pragma unroll
            for (int j = 0; j < 8; ++j) sum = energy_acc4(sum, yp[9 * s8 + j]);   // 8 float4 of data + 1 of padding per 32 samples
            if (VAD_WARPS == 2 && (s8 & 1)) between();                            // (a chain that may take two steps must serve fills more often)
        }
        if (VAD_WARPS == 1) between();
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) sum = energy_acc4(sum, yp[9 * 12 + j]);           // samples 384..399
    return __fdiv_rn(sum, (float)WIN);
}

// =============================================================================================
// role bodies
// =============================================================================================
__device__ __forceinline__ void role_fft(FusedSmem &sm, const FusedParams &P, int warp, int lane)
{
    const int l = lane & 15, half = lane >> 4;
    const int q = warp * 2 + half;                      // this half-warp's frame inside the step
    float *scr = sm.scr + warp * SCR_FLOATS_PER_WARP + 16 * half;
    const uint32_t tm = sm.tmem_base + ((uint32_t)(32 * ((threadIdx.x >> 5) & 3)) << 16);   // this (hardware) warp's lane quarter
    const bool on = P.n_mels != 0;
    AF_STATS_DECL
    // no tile state here: the resampler publishes what each step buffer holds (StepInfo), including the end of the work
    for (uint32_t it = 0;; ++it) {
        const int b = (int)(it & 1u);
        f2 R[8], I[8];
        AF_WAIT(&sm.y_full[b], (it >> 1) & 1u, 0);
        const int nv = sm.yinfo[b].n_valid;                 // frames that exist, STEP_LAST on the CTA's last step
        const bool work = on && warp * 2 < (nv & 0xff);     // warp-uniform: skip fully invalid pairs
        if (warp == 0 && lane == 0) sm.pinfo[it & 3u] = sm.yinfo[b];
        if (work) fft_load(sm.ybuf[b], tm, q, l, R, I);
        warp_arrive(&sm.y_empty[b], lane);                  // the step buffer (and its info) is no longer needed by this warp
        if (work) fft_passes(tm, scr, l, R, I);
        AF_WAIT(&sm.p_empty[b], ((it >> 1) & 1u) ^ 1u, 1);   // the mel warps are done with this power buffer
        if (work) fft_power(sm.pbuf[b], tm, q, l, lane, R, I);
        warp_arrive(&sm.p_full[b], lane);
        if (nv & STEP_LAST) break;
    }
    AF_STATS_FLUSH(0, lane);
}

// log2 of a value that is never subnormal (it was clamped to a normal floor): no range fix-up around MUFU.LG2
__device__ __forceinline__ float lg2_ftz(float x)
{
    float y;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// one step of a filter quad: four bins of each of the four filters against sixteen warp-uniform weights, all offsets
// immediate.  The weights come from tensor memory (one tcgen05.ld, issued before the power loads so that the two
// latencies overlap) or, for a quad that is not resident there, from shared memory.
#define AF_MEL_FMA16()                                                                              \
    a0 = fmaf(wa.x, xa.x, a0); a1 = fmaf(wa.y, xa.y, a1);                                         \
    b0 = fmaf(wb.x, xb.x, b0); b1 = fmaf(wb.y, xb.y, b1);                                         \
    c0 = fmaf(wc.x, xc.x, c0); c1 = fmaf(wc.y, xc.y, c1);                                         \
    d0 = fmaf(wd.x, xd.x, d0); d1 = fmaf(wd.y, xd.y, d1);                                         \
    a0 = fmaf(wa.z, xa.z, a0); a1 = fmaf(wa.w, xa.w, a1);                                         \
    b0 = fmaf(wb.z, xb.z, b0); b1 = fmaf(wb.w, xb.w, b1);                                         \
    c0 = fmaf(wc.z, xc.z, c0); c1 = fmaf(wc.w, xc.w, c1);                                         \
    d0 = fmaf(wd.z, xd.z, d0); d1 = fmaf(wd.w, xd.w, d1);
#define AF_MEL_STEP_S(i)                                                                            \
    {                                                                                               \
        const float4 wa = w4[4 * (i)], wb = w4[4 * (i) + 1], wc = w4[4 * (i) + 2], wd = w4[4 * (i) + 3]; \
        const float4 xa = pa[i], xb = pb[i], xc = pc[i], xd = pd[i];                                \
        AF_MEL_FMA16()                                                                              \
    }
#define AF_MEL_STEP_T(i)                                                                            \
    {                                                                                               \
        float w_[16];                                                                               \
        tmem_ld16(tq + 16u * (i), w_);                                                              \
        const float4 xa = pa[i], xb = pb[i], xc = pc[i], xd = pd[i];                                \
        tmem_wait_ld(w_);                                                                           \
        const float4 wa = make_float4(w_[0], w_[1], w_[2], w_[3]), wb = make_float4(w_[4], w_[5], w_[6], w_[7]);       \
        const float4 wc = make_float4(w_[8], w_[9], w_[10], w_[11]), wd = make_float4(w_[12], w_[13], w_[14], w_[15]); \
        AF_MEL_FMA16()                                                                              \
    }
// the steps run from the quad's last quadruple down to its first through an unrolled chain entered at `c4`
#define AF_MEL_CHAIN(STEP)                                                                          \
    switch (c4) {                                                                                   \
    case 8: STEP(7)                                                                                 \
    case 7: STEP(6)                                                                                 \
    case 6: STEP(5)                                                                                 \
    case 5: STEP(4)                                                                                 \
    case 4: STEP(3)                                                                                 \
    case 3: STEP(2)                                                                                 \
    case 2: STEP(1)                                                                                 \
    case 1: STEP(0)                                                                                 \
    default: break;                                                                                 \
    }

template <bool FAST_LOG, bool VEC>
__device__ __forceinline__ void role_mel_run(FusedSmem &sm, const FusedParams &P, int mw, int lane)
{
    const uint32_t M = P.n_mels;
    const float log_mul = P.log_scale, log_floor = P.log_floor;
    const int q0 = sm.mel.quad_begin[mw], q1 = sm.mel.quad_begin[mw + 1];
    const int fr = pb_frame(lane);                              // frame held by power row `lane`
    const uint32_t tm = sm.tmem_base + ((uint32_t)(32 * ((threadIdx.x >> 5) & 3)) << 16);   // this warp's lane quarter
    AF_STATS_DECL
    // no tile state here: the FFT warps forward what each power buffer holds (StepInfo), including the end of the work
    for (uint32_t it = 0;; ++it) {
        const int b = (int)(it & 1u);
        AF_WAIT(&sm.p_full[b], (it >> 1) & 1u, 0);
        const StepInfo info = sm.pinfo[it & 3u];
        const int n_valid = info.n_valid & 0xff;
        if (M && info.lm_dst && n_valid > 0) {
            const bool valid = fr < n_valid;
            float *dst = info.lm_dst + (uint32_t)fr * M + 4 * q0;
            const char *prow = reinterpret_cast<const char *>(sm.pbuf[b] + lane * PB_ROW);
            const uint4 *qtab = reinterpret_cast<const uint4 *>(&sm.mel.quad[q0]);
            for (int qd = q0; qd < q1; ++qd, qtab += 2, dst += 4) {
                const uint4 d0q = qtab[0], d1q = qtab[1];
                const float4 *pa = reinterpret_cast<const float4 *>(prow + d0q.x);
                const float4 *pb = reinterpret_cast<const float4 *>(prow + d0q.y);
                const float4 *pc = reinterpret_cast<const float4 *>(prow + d0q.z);
                const float4 *pd = reinterpret_cast<const float4 *>(prow + d0q.w);
                int c4 = (int)d1q.x;
                float a0 = 0.0f, a1 = 0.0f, b0 = 0.0f, b1 = 0.0f, c0 = 0.0f, c1 = 0.0f, d0 = 0.0f, d1 = 0.0f;
                if (d1q.z != MEL_NO_TMEM) {
                    const uint32_t tq = tm + d1q.z;
                    AF_MEL_CHAIN(AF_MEL_STEP_T)
                } else {
                    const float4 *w4 = reinterpret_cast<const float4 *>(reinterpret_cast<const char *>(sm.mel.w) + d1q.y);
#pragma unroll 1
                    for (; c4 > 8; --c4) AF_MEL_STEP_S(c4 - 1)      // wide filters (few mel bands): generic steps first
                    AF_MEL_CHAIN(AF_MEL_STEP_S)
                }
                float o[4];
                if (FAST_LOG) {
                    o[0] = lg2_ftz(fmaxf(a0 + a1, log_floor)) * log_mul;
                    o[1] = lg2_ftz(fmaxf(b0 + b1, log_floor)) * log_mul;
                    o[2] = lg2_ftz(fmaxf(c0 + c1, log_floor)) * log_mul;
                    o[3] = lg2_ftz(fmaxf(d0 + d1, log_floor)) * log_mul;
                } else {
                    o[0] = __log2f(fmaxf(a0 + a1, log_floor)) * log_mul;
                    o[1] = __log2f(fmaxf(b0 + b1, log_floor)) * log_mul;
                    o[2] = __log2f(fmaxf(c0 + c1, log_floor)) * log_mul;
                    o[3] = __log2f(fmaxf(d0 + d1, log_floor)) * log_mul;
                }
                if (valid) {
                    if (VEC) __stcs(reinterpret_cast<float4 *>(dst), make_float4(o[0], o[1], o[2], o[3]));
                    else {
#pragma unroll
                        for (int u = 0; u < 4; ++u)
                            if (4 * qd + u < (int)M) dst[u] = o[u];
                    }
                }
            }
        }
        warp_arrive(&sm.p_empty[b], lane);
        if (info.n_valid & STEP_LAST) break;
    }
    AF_STATS_FLUSH(1, lane);
}
#undef AF_MEL_CHAIN
#undef AF_MEL_STEP_T
#undef AF_MEL_STEP_S
#undef AF_MEL_FMA16

__device__ __forceinline__ void role_mel(FusedSmem &sm, const FusedParams &P, int mw, int lane)
{
    // the clamped value is normal: lg2.approx.ftz needs no range fix-up; 16-byte stores when every row allows them
    const bool fast_log = P.log_floor >= 1.17549435e-38f;
    const bool vec = (P.n_mels & 3u) == 0 && (P.logmel_stride & 3ull) == 0 && ((reinterpret_cast<uintptr_t>(P.logmel) & 15) == 0);
    if (fast_log && vec) role_mel_run<true, true>(sm, P, mw, lane);
    else if (vec) role_mel_run<false, true>(sm, P, mw, lane);
    else role_mel_run<false, false>(sm, P, mw, lane);
}

template <bool QUARTERS>
__device__ __forceinline__ void role_vad(FusedSmem &sm, const FusedParams &P, int lane, int vidx)
{
    // Two cursors.  FILLS (lane 0): the bulk copy of a half step is issued as soon as the resampler warps have
    // released its stage buffer -- blocking for the step the resamplers need next, and opportunistically (one
    // non-blocking test between the 128-sample segments of the energy chains) for the steps after it, so that a
    // long chain never delays a fill.  ENERGIES: the 32 frames of the previous step once its buffer is full.
    const bool chains = P.do_energy && P.energy;
    if (vidx != 0 && !chains) return;                       // a second V warp only takes energy chains (of the odd steps)
    AF_STATS_DECL
    // fill cursor (lane 0): tile, step, half.  The descriptors (source pointer, byte count, staged range) were planned
    // per tile on the host; the next one is fetched right after a fill is issued, so that issuing a fill is a
    // handful of instructions once its stage buffer is released.
    // The cursor counts PAIRS of fills (one per stage buffer): a step is one pair, or two when its input is staged in
    // quarters (fill[parts * step + part] = fill[2 * pair + half]), so a pair index works like the step index did.
    uint32_t tile_f = blockIdx.x, g_f = 0, it_f = 0, steps_f = 0;   // pair inside the tile, pairs issued so far, pairs of the tile
    int h_f = 0;
    bool fill_live = vidx == 0 && tile_f < P.n_tiles;
    FillDesc d_next{};
    auto fetch_desc = [&]() {
        const uint4 *src = reinterpret_cast<const uint4 *>(&P.tiles[tile_f].fill[2 * g_f + h_f]);
        const uint4 a = __ldg(src), b = __ldg(src + 1);
        d_next.src = reinterpret_cast<const char *>(((unsigned long long)a.y << 32) | a.x);
        d_next.bytes = a.z; d_next.lo = a.w; d_next.hi = b.x; d_next.interior = b.y;
    };
    auto tile_pairs = [&]() { return QUARTERS ? P.tiles[tile_f].n_steps * (P.tiles[tile_f].parts >> 1) : P.tiles[tile_f].n_steps; };
    if (lane == 0 && fill_live) { steps_f = tile_pairs(); fetch_desc(); }
    auto issue_next = [&](bool blocking) {                  // lane 0 only
        if (!fill_live) return;
        if (blocking) { AF_WAIT(&sm.stage_empty[h_f], (it_f & 1u) ^ 1u, 0); }
        else if (!mbar_test(&sm.stage_empty[h_f], (it_f & 1u) ^ 1u)) return;
        AF_TIC
        issue_fill(sm, P, d_next, h_f);
        if (++h_f == 2) {
            h_f = 0; ++it_f;
            if (++g_f == steps_f) {
                g_f = 0; tile_f += gridDim.x;
                fill_live = tile_f < P.n_tiles;
                if (fill_live) steps_f = tile_pairs();
            }
        }
        if (fill_live) fetch_desc();
        AF_TOC(2)
    };
    auto service = [&]() {
        if (lane == 0) issue_next(false);
        __syncwarp();
    };
    uint32_t it = 0, pairs_before = 0;                      // steps so far, and the fill pairs they took
    bool have_prev = false;
    uint32_t prev_f0 = 0, prev_nf = 0, prev_stream = 0, prev_it = 0;
    for (uint32_t tile = blockIdx.x;; tile += gridDim.x) {
        const bool live = tile < P.n_tiles;
        TileGeo t{};
        uint32_t n_frames = 0;
        if (live) t = tile_geo(P, tile, &n_frames);
        const uint32_t n_steps = live ? t.n_steps : 1u;        // one drain iteration after the last tile
        for (uint32_t g = 0; g < n_steps; ++g) {
            if (vidx == 0) {
                if (live) {
                    // the fills of the earlier steps and the first pair of step `it` are out (a second pair, if any, needs the
                    // resampler warps to release the buffers first: it goes out through service() or the next trip here)
                    if (lane == 0) while (fill_live && it_f <= pairs_before) issue_next(true);
                } else {
                    if (lane == 0) while (fill_live) issue_next(true);      // drain trip: the last step's later parts, if any
                }
                __syncwarp();
            }
            // with two V warps, V0 takes the even steps (ybuf[0]) and V1 the odd ones: a chain then has two steps of time
            if (have_prev && (VAD_WARPS == 1 || !chains || (prev_it & 1u) == (uint32_t)vidx)) {
                const int b = (int)(prev_it & 1u);
                AF_WAIT(&sm.y_full[b], (prev_it >> 1) & 1u, 1);
                if (chains) {
                    const int n_valid = prev_f0 < prev_nf ? (int)min((uint32_t)SF, prev_nf - prev_f0) : 0;
                    const float en = frame_energy_smem(sm.ybuf[b], lane, service);
                    if (lane < n_valid) P.energy[(uint64_t)prev_stream * P.energy_stride + prev_f0 + lane] = en;
                }
                warp_arrive(&sm.y_empty[b], lane);
            }
            if (live) {
                have_prev = true;
                prev_f0 = t.f_tile0 + g * SF; prev_nf = n_frames; prev_stream = t.stream; prev_it = it;
                ++it;
                pairs_before += QUARTERS ? (t.parts >> 1) : 1u;
            } else {
                have_prev = false;
            }
        }
        if (!live) break;
    }
    AF_STATS_FLUSH(2, lane);
}

#ifndef AF_FUSED_SPLIT_TU
// ---- R role, one loop for every kind of tile: the kernel all-48-kHz batches run (default translation unit).  Kept as it was when
// the two-instantiation loop below was introduced: the same logic wrapped differently compiles to a kernel that is 2-7 %
// slower on cfg2 (0.555 vs 0.565 / 0.595 ms measured), so the source of the fast one is left alone.
template <bool QUARTERS>
__device__ __forceinline__ void role_resample_single(FusedSmem &sm, const FusedParams &P, int rtid, int lane)
{
    uint32_t it = 0;
    uint32_t uses0 = 0;                                     // uses of EACH stage buffer before the current step (see role_vad: fills0)
    AF_STATS_DECL
    // the descriptor of a tile is fetched one tile ahead with cp.async into the warp's other slot (RsTile)
    const int w = rtid >> 5;
    auto prefetch = [&](uint32_t tile, int slot) {
        if (tile < P.n_tiles && lane < 7) {
            const char *src = reinterpret_cast<const char *>(P.tiles + tile) + (lane < 2 ? 16 * lane : (int)offsetof(TileDev, sdesc) + 16 * (lane - 2));
            cp_async16(reinterpret_cast<char *>(&sm.rs[slot][w]) + 16 * lane, src);
        }
    };
    int slot = 0;
    prefetch(blockIdx.x, 0);
    for (uint32_t tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x, slot ^= 1) {
        AF_TIC
        cp_async_wait_all();
        __syncwarp();                                   // the copy is visible to the warp; every lane is done with the other slot
        const RsTile &rt = sm.rs[slot][w];
        prefetch(tile + gridDim.x, slot ^ 1);
        TileGeo t;
        t.stream = rt.stream_idx; t.n_tile0 = rt.tile * TILE_SAMPLES; t.tile_end = rt.tile_end; t.n_steps = rt.n_steps;
        t.n_frames = rt.n_frames; t.parts = rt.parts;
        AF_TOC(2)
        const StreamDev &s = rt.stream;
        int kind = K_GENERIC;
        if (s.channels == 1) kind = s.format == FMT_F32 ? K_F32_1 : K_I16_1;
        else if (s.channels == 2) kind = s.format == FMT_F32 ? K_F32_2 : K_I16_2;
        float *pcm_row = P.pcm ? P.pcm + (uint64_t)t.stream * P.pcm_stride : nullptr;
        // does this tile's fast path hand out output quads to fixed owner threads (see resample_half_fast)?
        const bool quad_tile = s.mode != RS_PASSTHROUGH && ((kind == K_F32_1 && s.q == 1 && s.p == 3) || (kind != K_GENERIC && s.q > 1));
        bool prev_quads = false;
        // the hot case -- 48 kHz mono f32 -- bypasses the format dispatch: its interior half steps go straight to the quad loop
        const bool hot = kind == K_F32_1 && s.mode != RS_PASSTHROUGH && s.q == 1 && s.p == 3;
        const int tile_k = rt.tile_k;
        // parts per step: a compile-time 2 in the kernel instance for batches without quarter-staged streams
        const uint32_t parts = QUARTERS ? t.parts : 2u;

        for (uint32_t g = 0; g < t.n_steps; ++g, ++it) {
            const int b = (int)(it & 1u);
            const uint32_t toff = g * STEP_SAMPLES;
            YSink out{sm.ybuf[b], pcm_row, t.n_tile0 + toff, t.tile_end, P.neg_zero};
            const int lim4 = pcm_row ? (int)min((uint32_t)YLEN, out.wr_end - min(out.wr_end, out.base)) - 4 : -(1 << 30);
            AF_WAIT(&sm.y_empty[b], ((it >> 1) & 1u) ^ 1u, 0);   // FFT and VAD warps are done with this buffer
            AF_TIC2
            if (g > 0) {
                // the 240-sample overlap with the previous step
                const float *prev = sm.ybuf[b ^ 1];
                if (prev_quads) {
                    // the quad paths give every output quad a fixed owner thread: each thread carries the quad it wrote
                    // itself in the previous step -- no synchronisation among the resampler warps
                    constexpr int QS = 4 * RS_THREADS;
                    int c4 = LAST_PART_LO2 + 4 * rtid;
                    c4 += ((STEP_SAMPLES - c4 + QS - 1) / QS) * QS;           // first own quad at or after STEP_SAMPLES
                    if (c4 < YLEN)
                        *reinterpret_cast<float4 *>(out.yb + ypad(c4 - STEP_SAMPLES)) = *reinterpret_cast<const float4 *>(prev + ypad(c4));
                } else {
                    named_bar_sync(1, RS_THREADS);                            // written by all resampler threads: sync first
                    for (int i = rtid; i < CARRY; i += RS_THREADS) out.yb[ypad(i)] = prev[ypad(STEP_SAMPLES + i)];
                }
            }
            AF_TOC(3)
#pragma unroll 1
            for (int k = 0; k < (int)parts; ++k) {
                const int h = k & 1;                            // parts alternate between the two stage buffers
                AF_WAIT(&sm.stage_full[h], (uses0 + ((uint32_t)k >> 1)) & 1u, 1);
                const int i_lo = part_lo(g, (int)parts, k), i_hi = part_end((int)parts, k);
                AF_TIC2
                if (hot && sm.st_interior[h] == 1u) {
                    resample_quads_48k(reinterpret_cast<const float *>(sm.stage[h]) + (tile_k + 3 * (int)toff - 1 - (int)(uint32_t)sm.st_lo[h]),
                                       out.yb, out.pcm + out.base, lim4, i_lo, i_hi, rtid);
                } else {
                    switch (kind) {
                    case K_F32_1: resample_dispatch<K_F32_1>(sm, rt, h, s, out, toff, i_lo, i_hi, rtid); break;
                    case K_I16_1: resample_dispatch<K_I16_1>(sm, rt, h, s, out, toff, i_lo, i_hi, rtid); break;
                    case K_F32_2: resample_dispatch<K_F32_2>(sm, rt, h, s, out, toff, i_lo, i_hi, rtid); break;
                    case K_I16_2: resample_dispatch<K_I16_2>(sm, rt, h, s, out, toff, i_lo, i_hi, rtid); break;
                    default: resample_dispatch<K_GENERIC>(sm, rt, h, s, out, toff, i_lo, i_hi, rtid); break;
                    }
                }
                AF_TOC(4)
                if (k == (int)parts - 1) prev_quads = quad_tile && parts == 2u && sm.st_interior[1] != 0u;   // (read before the stage is released)
                warp_arrive(&sm.stage_empty[h], lane);          // this warp no longer reads stage[h] or its metadata
            }
            if (rtid == 0) {
                // what this step buffer holds, for the FFT and mel warps (they keep no tile state)
                const uint32_t f0 = (t.n_tile0 / HOP) + g * SF, n_frames = t.n_frames;
                StepInfo info;
                info.lm_dst = (P.logmel && P.n_mels) ? P.logmel + (uint64_t)t.stream * P.logmel_stride + (uint64_t)f0 * P.n_mels : nullptr;
                info.n_valid = f0 < n_frames ? (int)min((uint32_t)SF, n_frames - f0) : 0;
                if (g + 1 == t.n_steps && tile + gridDim.x >= P.n_tiles) info.n_valid |= STEP_LAST;
                info.pad_ = 0;
                sm.yinfo[b] = info;
            }
            warp_arrive(&sm.y_full[b], lane);
            uses0 += parts >> 1;
        }
    }
    AF_STATS_FLUSH(3, lane);
}

#else
// ---- R role for batches that also hold other tiles than 48 kHz mono f32 (-DAF_FUSED_SPLIT_TU) ----
template <bool QUARTERS>
__device__ __forceinline__ void role_resample_split(FusedSmem &sm, const FusedParams &P, int rtid, int lane)
{
    uint32_t it = 0;
    uint32_t uses0 = 0;                                     // uses of EACH stage buffer before the current step (see role_vad: fills0)
    AF_STATS_DECL
    // the descriptor of a tile is fetched one tile ahead with cp.async into the warp's other slot (RsTile)
    const int w = rtid >> 5;
    auto prefetch = [&](uint32_t tile, int slot) {
        if (tile < P.n_tiles && lane < 7) {
            const char *src = reinterpret_cast<const char *>(P.tiles + tile) + (lane < 2 ? 16 * lane : (int)offsetof(TileDev, sdesc) + 16 * (lane - 2));
            cp_async16(reinterpret_cast<char *>(&sm.rs[slot][w]) + 16 * lane, src);
        }
    };
    int slot = 0;
    prefetch(blockIdx.x, 0);
    for (uint32_t tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x, slot ^= 1) {
        AF_TIC
        cp_async_wait_all();
        __syncwarp();                                   // the copy is visible to the warp; every lane is done with the other slot
        const RsTile &rt = sm.rs[slot][w];
        prefetch(tile + gridDim.x, slot ^ 1);
        TileGeo t;
        t.stream = rt.stream_idx; t.n_tile0 = rt.tile * TILE_SAMPLES; t.tile_end = rt.tile_end; t.n_steps = rt.n_steps;
        t.n_frames = rt.n_frames; t.parts = rt.parts;
        AF_TOC(2)
        const StreamDev &s = rt.stream;
        int kind = K_GENERIC;
        if (s.channels == 1) kind = s.format == FMT_F32 ? K_F32_1 : K_I16_1;
        else if (s.channels == 2) kind = s.format == FMT_F32 ? K_F32_2 : K_I16_2;
        float *pcm_row = P.pcm ? P.pcm + (uint64_t)t.stream * P.pcm_stride : nullptr;
        // does this tile's fast path hand out output quads to fixed owner threads (see resample_half_fast)?
        // 48 kHz stereo f32 (cfg4): its staged interior parts take a quad loop of their own
        const bool hot2 = kind == K_F32_2 && s.mode != RS_PASSTHROUGH && s.q == 1 && s.p == 3;
        const bool quad_tile = s.mode != RS_PASSTHROUGH && ((kind == K_F32_1 && s.q == 1 && s.p == 3) || (kind != K_GENERIC && s.q > 1));
        bool prev_quads = false;
        // the hot case -- 48 kHz mono f32 -- bypasses the format dispatch: its interior half steps go straight to the quad loop
        const bool hot = kind == K_F32_1 && s.mode != RS_PASSTHROUGH && s.q == 1 && s.p == 3;
        const int tile_k = rt.tile_k;
        // parts per step: a compile-time 2 in the kernel instance for batches without quarter-staged streams
        const uint32_t parts = QUARTERS ? t.parts : 2u;

        // The steps of the tile, instantiated twice: HOT = 48 kHz mono f32 (its interior parts go straight to the quad loop and
        // nothing of the other formats is in the loop), and everything else.  In one shared loop the general path paid --
        // through register allocation -- for the hot one and the other way round (cfg3 13.1 -> 12.4 ms).
        auto run_steps = [&](auto hot_tag) {
        constexpr bool HOT = decltype(hot_tag)::value;
        for (uint32_t g = 0; g < t.n_steps; ++g, ++it) {
            const int b = (int)(it & 1u);
            const uint32_t toff = g * STEP_SAMPLES;
            YSink out{sm.ybuf[b], pcm_row, t.n_tile0 + toff, t.tile_end, P.neg_zero};
            const int lim4 = pcm_row ? (int)min((uint32_t)YLEN, out.wr_end - min(out.wr_end, out.base)) - 4 : -(1 << 30);
            AF_WAIT(&sm.y_empty[b], ((it >> 1) & 1u) ^ 1u, 0);   // FFT and VAD warps are done with this buffer
            AF_TIC2
            if (g > 0) {
                // the 240-sample overlap with the previous step
                const float *prev = sm.ybuf[b ^ 1];
                if (prev_quads) {
                    // the quad paths give every output quad a fixed owner thread: each thread carries the quad it wrote
                    // itself in the previous step -- no synchronisation among the resampler warps
                    constexpr int QS = 4 * RS_THREADS;
                    int c4 = (parts == 4u ? part_end(4, 2) : LAST_PART_LO2) + 4 * rtid;   // first quad of the step's last part
                    c4 += ((STEP_SAMPLES - c4 + QS - 1) / QS) * QS;           // first own quad at or after STEP_SAMPLES
                    if (c4 < YLEN)
                        *reinterpret_cast<float4 *>(out.yb + ypad(c4 - STEP_SAMPLES)) = *reinterpret_cast<const float4 *>(prev + ypad(c4));
                } else {
                    named_bar_sync(1, RS_THREADS);                            // written by all resampler threads: sync first
                    for (int i = rtid; i < CARRY; i += RS_THREADS) out.yb[ypad(i)] = prev[ypad(STEP_SAMPLES + i)];
                }
            }
            AF_TOC(3)
#pragma unroll 1
            for (int k = 0; k < (int)parts; ++k) {
                const int h = k & 1;                            // parts alternate between the two stage buffers
                const int i_lo = part_lo(g, (int)parts, k), i_hi = part_end((int)parts, k);
                AF_WAIT(&sm.stage_full[h], (uses0 + ((uint32_t)k >> 1)) & 1u, 1);
                AF_TIC2
                if (!HOT && hot2 && sm.st_interior[h] == 1u) {
                    resample_quads_48k_stereo(reinterpret_cast<const float *>(sm.stage[h]) +
                                                  2 * (tile_k + 3 * (int)toff - 1 - (int)((uint32_t)sm.st_lo[h] >> 1)),
                                              out.yb, out.pcm + out.base, lim4, i_lo, i_hi, rtid);
                } else if (HOT && sm.st_interior[h] == 1u) {
                    resample_quads_48k(reinterpret_cast<const float *>(sm.stage[h]) + (tile_k + 3 * (int)toff - 1 - (int)(uint32_t)sm.st_lo[h]),
                                       out.yb, out.pcm + out.base, lim4, i_lo, i_hi, rtid);
                } else if (HOT) {
                    resample_dispatch<K_F32_1>(sm, rt, h, s, out, toff, i_lo, i_hi, rtid);
                } else {
                    switch (kind) {
                    case K_F32_1: resample_dispatch<K_F32_1>(sm, rt, h, s, out, toff, i_lo, i_hi, rtid); break;
                    case K_I16_1: resample_dispatch<K_I16_1>(sm, rt, h, s, out, toff, i_lo, i_hi, rtid); break;
                    case K_F32_2: resample_dispatch<K_F32_2>(sm, rt, h, s, out, toff, i_lo, i_hi, rtid); break;
                    case K_I16_2: resample_dispatch<K_I16_2>(sm, rt, h, s, out, toff, i_lo, i_hi, rtid); break;
                    default: resample_dispatch<K_GENERIC>(sm, rt, h, s, out, toff, i_lo, i_hi, rtid); break;
                    }
                }
                AF_TOC(4)
                if (k == (int)parts - 1)                       // (read before the stage is released)
                    prev_quads = hot2 ? sm.st_interior[1] == 1u : (quad_tile && parts == 2u && sm.st_interior[1] != 0u);
                warp_arrive(&sm.stage_empty[h], lane);          // this warp no longer reads stage[h] or its metadata
            }
            if (rtid == 0) {
                // what this step buffer holds, for the FFT and mel warps (they keep no tile state)
                const uint32_t f0 = (t.n_tile0 / HOP) + g * SF, n_frames = t.n_frames;
                StepInfo info;
                info.lm_dst = (P.logmel && P.n_mels) ? P.logmel + (uint64_t)t.stream * P.logmel_stride + (uint64_t)f0 * P.n_mels : nullptr;
                info.n_valid = f0 < n_frames ? (int)min((uint32_t)SF, n_frames - f0) : 0;
                if (g + 1 == t.n_steps && tile + gridDim.x >= P.n_tiles) info.n_valid |= STEP_LAST;
                info.pad_ = 0;
                sm.yinfo[b] = info;
            }
            warp_arrive(&sm.y_full[b], lane);
            uses0 += parts >> 1;
        }
        };
        if (hot) run_steps(std::true_type{});
        else run_steps(std::false_type{});
    }
    AF_STATS_FLUSH(3, lane);
}

#endif

// QUARTERS: some stream of the batch stages its input in quarter steps (f32 stereo); the other instance keeps the
// two-parts-per-step constants folded in (measured: the general one costs mono batches 1.4 %, 2.8 % with the VAD on)
template <bool QUARTERS>
__global__ void __launch_bounds__(FUSED_THREADS, 1) af_fused_kernel(const FusedParams P)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    FusedSmem &sm = *reinterpret_cast<FusedSmem *>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    // constant tables -> shared memory, barriers (once per CTA)
    {
        if (P.n_mels) {
            const uint32_t *ms = reinterpret_cast<const uint32_t *>(P.mel);
            uint32_t *md = reinterpret_cast<uint32_t *>(&sm.mel);
            for (int i = tid; i < (int)(sizeof(MelTables) / 4); i += FUSED_THREADS) md[i] = ms[i];
        }
        for (int i = tid; i < 2 * PBUF_FLOATS; i += FUSED_THREADS) sm.pbuf[0][i] = 0.0f;
        if (P.per_q) {
            for (uint32_t r = tid; r < P.per_q; r += FUSED_THREADS) sm.koff[r] = (uint16_t)(((r + 1u) * P.per_p) / P.per_q);
        }
        if (tid == 0) {
            constexpr uint32_t QS = 4u * RS_THREADS;
            sm.per_p = P.per_p; sm.per_q = P.per_q;
            sm.sw_r = P.per_q ? QS % P.per_q : 0u;
            sm.sw_kp = P.per_q ? (QS / P.per_q) * P.per_p : 0u;
        }
    }
    if (tid == 0) {
        for (int h = 0; h < N_STAGE; ++h) {
            mbar_init(&sm.stage_full[h], 1);
            mbar_init(&sm.stage_empty[h], RS_WARPS);
        }
        for (int h = 0; h < 2; ++h) {
            mbar_init(&sm.y_full[h], RS_WARPS);
            mbar_init(&sm.y_empty[h], FFT_WARPS + 1);
        }
        for (int h = 0; h < 2; ++h) {
            mbar_init(&sm.p_full[h], FFT_WARPS);
            mbar_init(&sm.p_empty[h], MEL_WARPS);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) tmem_alloc(&sm.tmem_base);
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    if (warp < 4) {
        // warps 0..3 own the four TMEM lane quarters: thread t writes the constants of FFT lane l = t & 15 into its lane
        const uint32_t tm = sm.tmem_base + ((uint32_t)(32 * warp) << 16);
        const int l = lane & 15;
#pragma unroll
        for (int p = 0; p < 8; ++p) tmem_st4(tm + TM_TW1 + 4 * p, P.fft->tw1p[p * 16 + l]);
#pragma unroll
        for (int r = 0; r < 4; ++r) tmem_st4(tm + TM_TW2 + 4 * r, P.fft->tw2p[r * 16 + l]);
#pragma unroll
        for (int n1 = 0; n1 < 13; ++n1) tmem_st2(tm + TM_WIN + 2 * n1, P.fft->window[32 * n1 + 2 * l], P.fft->window[32 * n1 + 2 * l + 1]);
        tmem_wait_st();
    } else if (warp_role(P.layout, warp).role == ROLE_M && P.n_mels) {
        // every mel warp copies the weights of its resident quads into its own TMEM lane quarter: all 32 lanes (rows)
        // hold the same sixteen values per step, so that a 32x32b load hands every lane the warp-uniform weights
        const uint32_t tm = sm.tmem_base + ((uint32_t)(32 * (warp & 3)) << 16);
        const int mw = warp_role(P.layout, warp).index;
        for (int qd = sm.mel.quad_begin[mw]; qd < sm.mel.quad_begin[mw + 1]; ++qd) {
            const MelQuad &Q = sm.mel.quad[qd];
            if (Q.tcol == MEL_NO_TMEM) continue;
            const float4 *w4 = reinterpret_cast<const float4 *>(reinterpret_cast<const char *>(sm.mel.w) + Q.woff);
            for (uint32_t j = 0; j < Q.c4; ++j) tmem_st16(tm + Q.tcol + 16u * j, w4[4 * j], w4[4 * j + 1], w4[4 * j + 2], w4[4 * j + 3]);
        }
        tmem_wait_st();
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

    // 896 threads x 72 registers: every role fits (or nearly fits) that budget, so no setmaxnreg rebalancing
    const WarpRole wr = warp_role(P.layout, warp);
    if (wr.role == ROLE_F) role_fft(sm, P, wr.index, lane);
    else if (wr.role == ROLE_M) role_mel(sm, P, wr.index, lane);
    else if (wr.role == ROLE_V) role_vad<QUARTERS>(sm, P, lane, wr.index);
#ifdef AF_FUSED_SPLIT_TU
    else role_resample_split<QUARTERS>(sm, P, wr.index * 32 + lane, lane);
#else
    else role_resample_single<QUARTERS>(sm, P, wr.index * 32 + lane, lane);
#endif

    // every role has drained its pipeline: release the tensor memory
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) tmem_dealloc(sm.tmem_base);
}

#ifndef AF_FUSED_SPLIT_TU
size_t fused_smem_bytes() { return sizeof(FusedSmem); }
#endif

// debugging aid: copies (and clears) the pipeline statistics of both kernels; all zero unless built with -DAF_PIPE_STATS
#ifdef AF_FUSED_SPLIT_TU
cudaError_t fused_pipe_stats_split(unsigned long long out[32])
#else
static cudaError_t fused_pipe_stats_own(unsigned long long out[32])
#endif
{
#ifdef AF_PIPE_STATS
    cudaError_t e = cudaMemcpyFromSymbol(out, g_pipe_stats, sizeof(unsigned long long) * 32);
    if (e != cudaSuccess) return e;
    unsigned long long zero[32] = {};
    return cudaMemcpyToSymbol(g_pipe_stats, zero, sizeof(zero));
#else
    for (int i = 0; i < 32; ++i) out[i] = 0;
    return cudaSuccess;
#endif
}
#ifndef AF_FUSED_SPLIT_TU
cudaError_t fused_pipe_stats(unsigned long long out[32])
{
    unsigned long long other[32];
    cudaError_t e = fused_pipe_stats_own(out);
    if (e == cudaSuccess) e = fused_pipe_stats_split(other);
    for (int i = 0; i < 32 && e == cudaSuccess; ++i) out[i] += other[i];
    return e;
}
#endif

// the shared-memory attribute is per device: one flag per GPU of the process (af_init_multi drives several from one process)
template <class K>
static cudaError_t fused_attr(K kernel)
{
    return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(FusedSmem));
}

#ifdef AF_FUSED_SPLIT_TU
cudaError_t launch_fused_split(const FusedParams &P, int n_ctas, cudaStream_t st)
{
    static std::atomic<bool> attr_set[AF_MAX_GPUS_INTERNAL] = {};
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= AF_MAX_GPUS_INTERNAL) return cudaErrorInvalidDevice;
    if (!attr_set[dev].load(std::memory_order_acquire)) {
        e = fused_attr(af_fused_kernel<false>);
        if (e == cudaSuccess) e = fused_attr(af_fused_kernel<true>);
        if (e != cudaSuccess) return e;
        attr_set[dev].store(true, std::memory_order_release);
    }
    if (P.quarters) af_fused_kernel<true><<<n_ctas, FUSED_THREADS, sizeof(FusedSmem), st>>>(P);
    else af_fused_kernel<false><<<n_ctas, FUSED_THREADS, sizeof(FusedSmem), st>>>(P);
    return cudaGetLastError();
}
#else
cudaError_t launch_fused(const FusedParams &P, int n_ctas, cudaStream_t st, bool split)
{
    if (split || P.quarters) return launch_fused_split(P, n_ctas, st);
    static std::atomic<bool> attr_set[AF_MAX_GPUS_INTERNAL] = {};
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= AF_MAX_GPUS_INTERNAL) return cudaErrorInvalidDevice;
    if (!attr_set[dev].load(std::memory_order_acquire)) {
        e = fused_attr(af_fused_kernel<false>);
        if (e != cudaSuccess) return e;
        attr_set[dev].store(true, std::memory_order_release);
    }
    af_fused_kernel<false><<<n_ctas, FUSED_THREADS, sizeof(FusedSmem), st>>>(P);
    return cudaGetLastError();
}
#endif

}  // namespace af
