// af_common.cuh -- constants and device-visible tables shared by the kernels and the host runtime.
#pragma once
#include <cstddef>
#include <cstdint>
#include <cuda_runtime.h>

namespace af {

// ---- feature geometry (DESIGN.md "Feature spec"; absent from the reference, SURVEY R5) ----
constexpr int OUT_RATE = 16000;
constexpr int WIN = 400;          // 25 ms @ 16 kHz
constexpr int HOP = 160;          // 10 ms
constexpr int NFFT = 512;
constexpr int NBIN = NFFT / 2 + 1;   // 257
constexpr int MAX_MELS = 128;

// ---- reference resampler geometry (resampler.rs:47,55; rubato FastFixedIn) ----
constexpr int RS_CHUNK = 128;     // chunk_size
constexpr int RS_POLY = 8;        // rubato POLYNOMIAL_LEN

// ---- fused kernel tiling (one persistent CTA per SM, warp-specialised pipeline) ----
constexpr int SF = 32;                       // frames per step: one per half-warp of the 16 FFT warps
constexpr int STEP_SAMPLES = SF * HOP;       // 5120 new 16 kHz samples per step
constexpr int CARRY = WIN - HOP;             // 240 samples shared with the next step
constexpr int YLEN = STEP_SAMPLES + CARRY;   // 5360 samples live per step
// A step's raw input is staged in PARTS fills that alternate between the two stage buffers: while the resampler warps
// work on one part the next fill is in flight.  Two parts per step when half a step of raw input fits a buffer (mono,
// i16 stereo), four when only a quarter does (f32 stereo at 48 kHz: 1344 outputs x 3 frames x 8 B = 32 256 B); the
// boundaries are multiples of 32 outputs (the padding phase of the step buffer).  Measured for mono (cfg2, same box):
// two parts 0.577 ms, three parts over three smaller buffers 0.607 ms -- the extra barrier round trip and part
// prologue per step cost more than the deeper prefetch gains.
constexpr int N_STAGE = 2;                   // stage buffers
constexpr int MAX_PARTS = 4;
__host__ __device__ constexpr int part_end(int parts, int k)   // outputs [part_end(k - 1), part_end(k)) of the step buffer form part k
{
    return parts == 4 ? (k == 0 ? 1344 : (k == 1 ? 2688 : (k == 2 ? 4032 : 5360))) : (k == 0 ? 2688 : 5360);
}
__host__ __device__ constexpr int part_max_out(int parts) { return parts == 4 ? 1344 : 2688; }   // most outputs one part produces
constexpr int LAST_PART_LO2 = 2688;          // first output of the last part of a two-part step (the quad paths run on those)
constexpr int TILE_FRAMES = 128;             // frames per tile (work unit of one CTA)
constexpr int TILE_SAMPLES = TILE_FRAMES * HOP;   // 20480
constexpr int FFT_WARPS = 16;                // "F": window + FFT + power, one frame per half-warp
constexpr int MEL_WARPS = 4;                 // "M": mel projection + log, lane = frame
#ifdef AF_V2
constexpr int VAD_WARPS = 2;
constexpr int RS_WARPS = 6;
#else
constexpr int VAD_WARPS = 1;
constexpr int RS_WARPS = 7;
#endif
constexpr int RS_WARPS_DOC = 7;                  // "R": downmix + resample + PCM write-out.  224 threads: a half step (2688
                                             // outputs) is exactly three quads per thread
constexpr int RS_THREADS = RS_WARPS * 32;
constexpr int FUSED_WARPS = FFT_WARPS + MEL_WARPS + VAD_WARPS + RS_WARPS;   // 28 (one "V" warp: stage fills + sequential frame energies)
constexpr int FUSED_THREADS = FUSED_WARPS * 32;   // 896
// Which role a hardware warp plays.  Warp w issues from scheduler (SM sub-partition) w % 4, seven warps each, and
// addresses TMEM lane quarter w % 4.  Three layouts, chosen per launch (FusedParams::layout):
//   0  balanced: four FFT warps per scheduler -- best with the VAD off (measured 0.580 vs 0.597 ms, cfg2)
//   1  the V warp, whose 400-term dependent chains are the critical path with the VAD on, shares its scheduler with
//      only two of the issue-hungry FFT warps (0.702 vs 0.750 ms)
//   2  ... with only one
//   3  ... with none (mel + five resampler warps)
// In every layout mel warp j sits on scheduler j, so the TMEM columns of the mel weights do not depend on the layout.
enum : int { ROLE_F = 0, ROLE_M = 1, ROLE_V = 2, ROLE_R = 3 };
constexpr int N_LAYOUTS = 4;
struct WarpRole { int role, index; };
constexpr unsigned long long pack_layout(int layout)
{
    constexpr int F = ROLE_F, M = ROLE_M, V = ROLE_V, R = ROLE_R;
    // rows = w / 4, columns = scheduler
#ifdef AF_V2
    constexpr int tab[N_LAYOUTS][FUSED_WARPS] = {
        {V, V, F, F,  M, M, M, M,  R, R, R, R,  R, R, F, F,  F, F, F, F,  F, F, F, F,  F, F, F, F},
        {V, V, F, F,  M, M, M, M,  R, R, R, R,  R, R, F, F,  F, F, F, F,  F, F, F, F,  F, F, F, F},
        {V, V, F, F,  M, M, M, M,  R, R, R, R,  R, R, F, F,  F, F, F, F,  F, F, F, F,  F, F, F, F},
        {V, V, F, F,  M, M, M, M,  R, R, R, R,  R, R, F, F,  F, F, F, F,  F, F, F, F,  F, F, F, F}};
#else
    constexpr int tab[N_LAYOUTS][FUSED_WARPS] = {
        {F, F, F, F,  F, F, F, F,  F, F, F, F,  F, F, F, F,  M, M, M, M,  V, R, R, R,  R, R, R, R},
        {V, F, F, F,  F, F, F, F,  F, F, F, F,  M, F, F, F,  R, M, M, M,  R, F, F, R,  R, R, R, R},
        {V, F, F, F,  F, F, F, F,  M, F, F, F,  R, M, M, M,  R, F, F, F,  R, F, F, F,  R, R, R, R},
        {V, F, F, F,  M, F, F, F,  R, F, F, F,  R, F, F, F,  R, F, F, F,  R, F, R, R,  R, M, M, M}};
#endif
    unsigned long long m = 0;
    for (int w = 0; w < FUSED_WARPS; ++w) m |= (unsigned long long)tab[layout][w] << (2 * w);
    return m;
}
// two bits per warp, so that the kernel decodes its role from an immediate (no table in local memory)
constexpr unsigned long long LAYOUT_BITS0 = pack_layout(0), LAYOUT_BITS1 = pack_layout(1), LAYOUT_BITS2 = pack_layout(2),
                             LAYOUT_BITS3 = pack_layout(3);
__host__ __device__ constexpr int warp_role_of(int layout, int w)
{
    const unsigned long long m = layout == 0 ? LAYOUT_BITS0 : (layout == 1 ? LAYOUT_BITS1 : (layout == 2 ? LAYOUT_BITS2 : LAYOUT_BITS3));
    return (int)((m >> (2 * w)) & 3ull);
}
__host__ __device__ constexpr WarpRole warp_role(int layout, int w)
{
    const int r = warp_role_of(layout, w);
    int idx = 0;
    for (int i = 0; i < w; ++i) idx += warp_role_of(layout, i) == r ? 1 : 0;
    return WarpRole{r, idx};
}
constexpr bool layouts_ok()
{
    for (int l = 0; l < N_LAYOUTS; ++l) {
        int n[4] = {0, 0, 0, 0};
        for (int w = 0; w < FUSED_WARPS; ++w) {
            const WarpRole r = warp_role(l, w);
            ++n[r.role];
            if (r.role == ROLE_M && (w & 3) != r.index) return false;      // mel warp j on scheduler / TMEM quarter j
        }
        if (n[ROLE_F] != FFT_WARPS || n[ROLE_M] != MEL_WARPS || n[ROLE_V] != VAD_WARPS || n[ROLE_R] != RS_WARPS) return false;
    }
    return true;
}
static_assert(layouts_ok(), "every layout needs 16 F, 4 M (mel warp j on scheduler j), 1 V and 7 R warps");

// padded index of 16 kHz sample i inside the step buffer: 4 pad words after every 32 samples so
// that the 32 VAD lanes (frame starts 160 apart) hit distinct bank quads with LDS.128
__host__ __device__ constexpr int ypad(int i) { return i + 4 * (i >> 5); }
constexpr int YBUF_FLOATS = ((ypad(YLEN + 32) + 31) / 32) * 32;

// transpose scratch of one FFT warp (two frames): element (half h, row k1, column c) at k1 * 36 + 16 h + c, so the two
// half-warps store to disjoint bank halves and the row reads (LDS.128) are conflict free; the real and the
// imaginary parts go through the same scratch in turn
constexpr int SCR_ROW = 36;
constexpr int SCR_FLOATS_PER_WARP = 16 * SCR_ROW;        // 576 floats = 2304 B
// power buffer of one step: one row of PB_ROW floats per frame (bins 0..256, then zeros that the 4-padded mel
// weights may touch), read by the mel warps with LDS.128 (lane = row).  Frame q = 2 w + h of FFT warp w sits in row
// pb_row(q): the two frames of a warp are 16 banks apart (conflict-free column stores) and eight consecutive rows
// start in distinct 16-byte bank groups (conflict-free LDS.128), because PB_ROW / 4 is odd.
constexpr int PB_ROW = 260;
constexpr int PB_COLS = PB_ROW;              // bins a padded weight quadruple may read: [0, PB_COLS)
constexpr int PBUF_FLOATS = SF * PB_ROW;
__host__ __device__ constexpr int pb_row(int q) { return ((q >> 1) & 3) + 8 * (q >> 3) + 4 * (q & 1); }
__host__ __device__ constexpr int pb_frame(int row) { return 2 * ((row & 3) + 4 * (row >> 3)) + ((row >> 2) & 1); }
constexpr int KOFF_MAX = 640;                // longest output period (q) the periodic-position path of the resampler serves
constexpr int STAGE_BYTES = 32384;           // one TMA-staged part of raw input (2688 outputs x 3 x 4 B + halo), two of them

// formats / flags (mirror include/audioflow_gpu.h)
enum : uint16_t { FMT_F32 = 0, FMT_I16 = 1 };

// one stream of a batch, device resident
struct StreamDev {
    const void *data;        // interleaved samples
    uint64_t n_samples;      // total interleaved samples
    uint32_t n_in;           // mono frames = ceil(n_samples / channels)
    uint32_t n_out;          // resampled length (BatchResampler all + flush)
    uint32_t n_frames;       // STFT frames
    uint32_t n_vad_frames;   // VAD frames
    uint16_t channels;
    uint16_t format;
    uint32_t p, q;           // input step per output = p / q (reduced)
    uint32_t mode;           // RS_*
    const float *frac;       // RS_TABLE: f32 fractional offsets by output index
    uint32_t tile_begin;     // first tile of this stream in planning order (batches launch them in balance_tile_order)
    uint32_t n_tiles;
    uint32_t staged;         // parts per step when the input is staged through shared memory (2 or 4); 0: it does not fit
                             // (taps come from global memory; the step still runs as two parts)
    uint32_t pad_;
};
enum : uint32_t { RS_PASSTHROUGH = 0, RS_EXACT = 1, RS_TABLE = 2 };

// one staged half step: what the V warp needs to issue its bulk copy and what the resampler warps need to read it
struct FillDesc {
    const char *src;         // first staged byte in global memory
    uint32_t bytes;          // 0: nothing staged (taps come from global memory)
    uint32_t lo, hi;         // interleaved element range [lo, hi) held by the stage (fits 32 bits: n_in < 2^31, <= 2 channels staged)
    uint32_t interior;       // 1: every tap of the half step is inside the stage and the stream; 2: inside the stream but not
                             // staged (unchecked global loads); 0: checked path
    uint32_t pad_[2];
};
constexpr int TILE_FILLS = MAX_PARTS * (TILE_FRAMES / SF);   // fill descriptors per tile (fill[parts * step + part])

// one tile (128 frames of one stream) with everything the kernel would otherwise have to derive with 64-bit
// divisions: planned once per batch on the host (plan_tile, af_device.cuh), or per tick by the session set-up kernel
struct alignas(16) TileDev {
    uint32_t stream;
    uint32_t tile;           // tile index inside the stream
    int32_t k0;              // floor(position) of the tile's first output, in input frames
    uint32_t rem0;           // and its remainder (numerator units)
    uint32_t n_steps;        // steps of 32 frames
    uint32_t tile_end;       // the tile owns stream samples [tile * TILE_SAMPLES, tile_end)
    uint32_t n_frames;       // STFT frames of the stream (copy)
    uint32_t parts;          // stage fills per step: 2 or 4 (fill[parts * step + part])
    FillDesc fill[TILE_FILLS];
    StreamDev sdesc;         // copy of the stream's descriptor: one level of loads per tile instead of two
    uint32_t inc_k, inc_rem; // position increment of RS_THREADS outputs: (RS_THREADS * p) / q and % q
};
static_assert(sizeof(FillDesc) == 32, "a fill descriptor is fetched with two 16-byte loads");
static_assert(sizeof(TileDev) % 16 == 0 && offsetof(TileDev, fill) % 16 == 0, "fill descriptors must be 16-byte aligned");

// mel filterbank in compact form (weights already carry the 1/4 of the unscaled power).  The mel warps work
// lane = frame and walk FOUR adjacent filters (a "quad": one 16-byte store per frame) at a time, eight
// independent FMA chains: the quad's weights are zero padded to a common number of quadruples and interleaved
// [a0..a3][b0..b3][c0..c3][d0..d3] per step.  The quads are split over the MEL_WARPS warps by cost.  The weights of
// a quad are warp-uniform: they are served from tensor memory (one tcgen05.ld of 16 columns per step, no
// shared-memory bandwidth) when the quarter of TMEM its warp can address has room for them, else by LDS.128.
struct alignas(16) MelQuad {
    uint32_t off[4];         // byte offset, inside a power row, of the first bin each of the four filters reads (a multiple of 16)
    uint32_t c4;             // number of weight quadruples per filter; off / 4 + 4 c4 <= PB_COLS
    uint32_t woff;           // byte offset of the quad's weights inside MelTables::w (a multiple of 64)
    uint32_t tcol;           // first TMEM column of the quad's weights (16 columns per step), MEL_NO_TMEM: not resident
    uint32_t pad_;
};
constexpr uint32_t MEL_NO_TMEM = 0xffffffffu;
constexpr uint32_t TMEM_COLS = 512;          // the whole tensor memory of the SM (one CTA per SM)
constexpr uint32_t TM_MEL0 = 80;             // first column of the mel weights (the FFT constants use 0..73)
struct MelTables {
    MelQuad quad[MAX_MELS / 4];
    uint16_t n_w;
    uint16_t n_mels;
    uint16_t quad_begin[MEL_WARPS + 1];   // mel warp j owns filter quads [quad_begin[j], quad_begin[j + 1])
    alignas(16) float w[1536];
};
static_assert(sizeof(MelQuad) == 32, "MelQuad is read with two LDS.128");
static_assert(offsetof(MelTables, w) % 16 == 0, "mel weights must be 16-byte aligned");

// what the roles downstream of the resampler need to know about a step (32 frames): published through shared
// memory with the buffer hand-off, so that the FFT and mel warps keep no tile state of their own
struct alignas(16) StepInfo {
    float *lm_dst;           // log-mel row of the step's first frame (nullptr: no features)
    int n_valid;             // low byte: frames of the step that exist in the stream (0..32); STEP_LAST: the CTA's last step
    uint32_t pad_;
};
constexpr int STEP_LAST = 0x100;

// constant tables of the FFT, filled by the host in f64 and rounded once
struct FftTables {
    float window[416];       // periodic Hann, zero beyond 400
    // twiddles in the layout of the packed (f32x2) FFT: one float4 = (re_a, re_b, im_a, im_b) for the two points a
    // pack holds.  tw1p[p * 16 + l]: exp(-2 pi i l k1 / 256) for the points in slots 2p, 2p+1 of the 16-point
    // transform (slot s holds k1 = (s >> 2) + 4 (s & 3)); tw2p[r * 16 + l]: exp(-2 pi i k / 512), k = l + 16 r and
    // k = l + 16 (r + 4).
    float4 tw1p[8 * 16];
    float4 tw2p[4 * 16];
};

struct VadParams {
    float alpha;             // smoothing_factor
    float e_min;             // smallest f32 energy with 20*log10f(e) > threshold_db (host libm); +inf if none
    unsigned long long silence_timeout;
    unsigned long long min_speech;
};

struct VadState {
    float smoothed;
    int state;
    unsigned long long silence_frames;
    unsigned long long speech_frames;
};

struct FusedParams {
    const StreamDev *streams;
    const TileDev *tiles;
    uint32_t n_tiles;
    const FftTables *fft;
    const MelTables *mel;
    float *pcm;   uint64_t pcm_stride;
    float *logmel; uint64_t logmel_stride;
    float *energy; uint64_t energy_stride;
    uint32_t n_mels;         // 0: skip STFT/mel
    uint32_t do_energy;      // VAD energies on the STFT frames
    float log_floor;
    float log_scale;         // ln(2) (natural log) or log10(2): multiplies log2(mel)
    uint32_t use_stage;      // 0: plain global loads everywhere ("sync" variant)
    uint32_t layout;         // warp-to-role layout (warp_role)
    uint32_t quarters;       // 1: some tile stages its input in quarter steps (TileDev::parts == 4): general kernel instance
    float neg_zero;          // -0.0f, unknown to the compiler: the addend of the packed cubic's products (interp_cubic2)
    uint32_t per_p, per_q;   // RS_TABLE streams with this p / q take the periodic-position path (resample_part_periodic); 0: none
};

}  // namespace af
