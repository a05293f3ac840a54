// af_launch.h -- host-callable launch wrappers implemented in the .cu files.
#pragma once
#include "af_common.cuh"

namespace af {

// one contiguous piece of a mono f32 device signal to resample (compat objects, sessions)
struct ResampleJob {
    const float *data;       // mono f32, data[0] is global input index data_base
    long long data_base;
    long long n_valid_end;   // global input indices >= this (and < data_base) read as 0
    unsigned long long n_begin, n_end;   // global output indices [n_begin, n_end)
    uint32_t p, q, mode;
    const float *frac;       // RS_TABLE: indexed by global output index
    float *out;              // out[n - n_begin]
};

struct EnergyJob {           // generic frame energies over a device signal
    const float *y;          // row base
    uint64_t y_stride;       // floats between streams
    const uint32_t *n_frames;   // per stream (device) or nullptr -> n_frames_all
    uint32_t n_frames_all;
    uint32_t frame_len, hop;
    float *energy; uint64_t energy_stride;
    uint32_t n_streams;
};

struct ScanRec {             // one stream's detector configuration (ScanJob::recs), 32 bytes
    VadParams prm;
    uint32_t warm;           // EMA warm-up of the parallel kernels, scan_warmup(prm.alpha)
    uint32_t seq;            // 1: the stream needs the sequential kernel (warm == 0, or counters beyond the 32-bit path)
};
ScanRec scan_rec(const VadParams &prm);

struct ScanJob {             // EMA + threshold + state machine, one stream per thread
    const float *energy; uint64_t energy_stride;
    const uint32_t *n_frames; uint32_t n_frames_all;
    uint8_t *states; uint64_t states_stride;      // may be nullptr
    VadState *state_io;      // per stream: initial state in, final state out (nullptr -> fresh)
    VadState *final_out;     // optional extra copy of the final state (af_vad_final layout)
    VadParams prm;
    uint32_t n_streams;
    // long streams (optional): an upper bound of the frame counts known on the host, and scratch of
    // scan_scratch_words(max_frames) 32-bit words per stream; with both set, streams longer than two scan blocks are
    // scanned by many CTAs each (launch_vad_scan picks the path)
    uint32_t max_frames;
    uint32_t *scratch;
    // per-stream configurations (optional, device): recs[s] replaces prm for stream s; n_seq of the records have seq set.
    // The parallel (or long) kernel runs over every stream and the sequential kernel follows for the flagged ones only
    const ScanRec *recs;
    uint32_t n_seq;
};
size_t scan_scratch_words(uint32_t max_frames);
// kernel launches launch_vad_scan enqueues for `job`, counting the three long-stream phases as one
uint32_t scan_launches(const ScanJob &job);

struct SessionIngest {
    const float *old_buf; float *new_buf; uint64_t buf_stride;   // mono f32 input history, ping-pong
    uint32_t drop, keep;                                         // retained frames: old[drop .. drop + keep)
    const void *input; uint64_t in_stride_bytes;                 // this tick's interleaved samples, one row per stream
    uint64_t n_samples; uint32_t n_new_frames; uint32_t channels, format;
};

struct SessionResample {
    const float *in_buf; uint64_t in_stride;
    long long data_base, n_valid_end;                            // global frame index of in_buf[0]; frames beyond read 0
    unsigned long long n_begin, n_end;                           // global output range of this tick
    uint32_t p, q, mode;
    const float *frac;                                           // RS_TABLE: frac[n - n_begin]
    const float *y_old; float *y_new; uint64_t y_stride;         // 16 kHz carry + new samples, ping-pong
    uint32_t y_drop, y_keep;
};

// one stream's part of a tick of independent stream timelines (af_session_push_streams), planned on the host; it
// overrides the per-stream fields of SessionIngest / SessionResample / WireJob and the peak's range.  flags >>
// TICK_FMT_SHIFT is the stream's index into the session's SessionFormat table (inside `flags`, so StreamTick keeps the
// 64-byte layout the peak and wire kernels index)
constexpr uint32_t TICK_RESTART = 1, TICK_END = 2, TICK_FMT_SHIFT = 16;
struct SessionFormat {       // one capture format a session admits: load_mono's channels, session_resample_one's ratio
    uint32_t channels, p, q, mode;
};
struct StreamTick {
    uint32_t in_drop, in_keep;                                   // ingest: retained frames old[in_drop .. in_drop + in_keep)
    uint32_t n_new, n_samples;                                   // this tick's frames / interleaved samples of the stream
    long long data_base, n_valid_end;                            // resample (an end: n_valid_end at the real end of the data)
    unsigned long long n_begin;
    uint32_t n_y, frac_off;                                      // 16 kHz samples of the tick; RS_TABLE: fractions at frac[frac_off]
    uint32_t y_drop, y_keep;                                     // carry: y_old[y_drop .. y_drop + y_keep); new samples at y_keep
    uint32_t T, flags;                                           // frames completed; TICK_RESTART (history zeroed, detector and
                                                                 // wire segment cleared first) | TICK_END
};

struct GateJob {             // VAD-gated compaction (all device pointers)
    const float *pcm; uint64_t pcm_stride;           // 16 kHz rows (or nullptr)
    const float *logmel; uint64_t logmel_stride;     // [frame][mel] rows (or nullptr)
    uint32_t n_mels, hop;
    const uint32_t *n_out;                           // per-stream PCM lengths (or nullptr: unchecked)
    const uint32_t *seg; uint32_t seg_cap; const uint32_t *n_seg;   // af_vad_segments output
    uint32_t *off;                                   // [n_streams][seg_cap + 1] compacted frame offset of every segment
    uint32_t *total;                                 // [n_streams] kept frames
    float *out_pcm; uint64_t out_pcm_stride;
    float *out_lm; uint64_t out_lm_stride;
    uint32_t n_streams;
};
cudaError_t launch_vad_gate(const GateJob &job, cudaStream_t st);

struct WireTick {            // af_wire_tick (static_assert'ed in af_runtime.cu)
    uint32_t n_samples, n_chars, continued;
    uint16_t started, ended;
    uint8_t in_speech, pad[3];
};

struct WireJob {             // a session tick's wire payloads (all device pointers)
    const float *y; uint64_t y_stride;               // 16 kHz rows: frame f of the tick starts at y[f * hop]
    uint32_t y_new, n_new;                           // the tick's new samples are y[y_new, y_new + n_new)
    const uint8_t *states; uint64_t st_stride;       // VadState of the tick's T frames (nullptr: no VAD, or T == 0)
    uint32_t T, hop, gate;
    uint8_t *prev;                                   // per stream: state of the latest completed frame, carried across ticks
    int16_t *pcm16; uint64_t pcm16_stride;           // (or nullptr)
    char *b64; uint64_t b64_stride;                  // (or nullptr; stride a multiple of 4)
    WireTick *ticks;
    uint32_t n_streams;
    const StreamTick *tab;                           // ragged tick: per-stream y_new / n_new / T and the end flag (or nullptr)
};
cudaError_t launch_session_wire(const WireJob &job, cudaStream_t st);

size_t fused_smem_bytes();
cudaError_t fused_pipe_stats(unsigned long long out[32]);
cudaError_t launch_session_tick(const SessionIngest &I, const SessionResample &R, uint32_t n_streams, cudaStream_t st);
// the same with every stream planned by its own StreamTick, in its own format fmts[tab[s].flags >> TICK_FMT_SHIFT];
// restarted streams clear vad[s] and (if non-null) wire_prev[s]; pcm (device, or nullptr) receives each stream's new
// samples at its row start
cudaError_t launch_session_tick_streams(const SessionIngest &I, const SessionResample &R, const StreamTick *tab,
                                        const SessionFormat *fmts, VadState *vad, uint8_t *wire_prev, float *pcm,
                                        uint64_t pcm_stride, uint32_t n_streams, cudaStream_t st);
// split: the batch holds tiles other than 48 kHz mono f32 -> 16 kHz; such batches (and quarter-staged ones) run the
// kernel of the second translation unit of af_fused.cu (AF_FUSED_SPLIT_TU), whose resampler role keeps the hot and the
// general tiles in separate loops
cudaError_t launch_fused(const FusedParams &P, int n_ctas, cudaStream_t st, bool split = false);
cudaError_t launch_fused_split(const FusedParams &P, int n_ctas, cudaStream_t st);
cudaError_t fused_pipe_stats_split(unsigned long long out[32]);
// tab (or nullptr): stream s covers y[tab[s].y_keep, + tab[s].n_y) of its row instead of y[0, n)
cudaError_t launch_peak(const float *y, uint64_t y_stride, uint32_t n, uint32_t n_streams, float *peak, cudaStream_t st,
                        const StreamTick *tab = nullptr);

cudaError_t launch_to_mono(const float *in, uint64_t n_samples, uint32_t channels, float *out, uint64_t n_frames,
                           cudaStream_t st);
cudaError_t launch_resample_jobs(const ResampleJob *jobs_dev, uint32_t n_jobs, uint32_t max_outputs, cudaStream_t st);
cudaError_t launch_frame_energy(const EnergyJob &job, cudaStream_t st);
cudaError_t launch_vad_scan(const ScanJob &job, cudaStream_t st);   // (scan_launches above)
cudaError_t launch_pcm16(const float *in, uint64_t n, int16_t *out, cudaStream_t st);
cudaError_t launch_pcm16_base64(const float *in, uint64_t n, char *out, cudaStream_t st);   // 4 * ceil(2 n / 3) characters
cudaError_t launch_pcm16_rows(const float *in, uint64_t in_stride, int16_t *out, uint64_t out_stride, uint32_t width, uint32_t rows,
                              cudaStream_t st);
cudaError_t launch_vad_segments(const uint8_t *states, uint64_t stride, const uint32_t *n_frames, uint32_t n_streams,
                                uint32_t *seg, uint32_t seg_cap, uint32_t *n_seg, cudaStream_t st);

}  // namespace af
