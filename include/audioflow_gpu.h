/*
 * audioflow_gpu.h -- C ABI of libaudioflow_gpu.so, the B200 (sm_100a) implementation of the
 * audio hot path of forfd8960/audio-flow-rs:
 *
 *     interleaved f32/i16 PCM -> downmix -> resample to 16 kHz -> 25 ms/10 ms frames
 *     -> Hann -> 512-pt STFT -> log-mel,  and energy VAD frame decisions.
 *
 * Every entry point names the reference interface it replaces (paths relative to the
 * reference repo root).  The reference has no FFI of its own (plain Rust structs re-exported
 * at src-tauri/src/modules/audio/mod.rs:9-11), so these are exactly the functions a Rust
 * `extern "C"` block for that module would bind; INTEGRATION.md shows that binding.
 *
 * Conventions
 *   - plain C types only; every function returns an af_status (0 = ok) unless noted.
 *   - on failure a thread-local message is available from af_last_error(); the Rust shim
 *     turns it into AudioError::ResamplingFailed(msg) (src-tauri/src/error.rs:109-110).
 *   - handles are NOT thread-safe individually (they mirror `&mut self`); distinct handles
 *     may be used from distinct threads.
 *   - there is no CPU fallback: without a CUDA device every call fails with AF_ERR_NO_DEVICE.
 */
#ifndef AUDIOFLOW_GPU_H
#define AUDIOFLOW_GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define AF_API __attribute__((visibility("default")))
#else
#define AF_API
#endif

typedef enum af_status {
    AF_OK = 0,
    AF_ERR_INVALID = 1,           /* bad argument */
    AF_ERR_RESAMPLING_FAILED = 2, /* AudioError::ResamplingFailed (error.rs:109-110) */
    AF_ERR_CUDA = 3,              /* CUDA runtime failure (also surfaced as ResamplingFailed by the shim) */
    AF_ERR_NO_DEVICE = 4,         /* no CUDA device / not initialised */
    AF_ERR_CAPACITY = 5           /* caller-provided output buffer too small */
} af_status;

/* ---- library ------------------------------------------------------------------------- */
#define AF_MAX_GPUS 16
/* Selects GPU `device` for the calling THREAD, initialising the library's context on it at first use (device < 0:
 * keep the thread's selection / the process default).  A process may use several GPUs: objects remember the GPU they
 * were created on and every call that takes a handle runs there, whatever the calling thread has selected. */
AF_API int af_init(int device);
AF_API int af_current_device(void);             /* the calling thread's GPU, -1 before any af_init */
/* Makes `cuda_stream` (a cudaStream_t) the stream the library enqueues on for the calling thread's GPU wherever an
 * entry point has no stream argument of its own (sessions, sharded batches, the NULL-stream form of af_batch_run);
 * NULL restores the library's own non-blocking stream.  The caller keeps the stream alive. */
AF_API int af_set_stream(void *cuda_stream);
AF_API int af_shutdown(void);
AF_API size_t af_last_error(char *buf, size_t cap);   /* returns strlen of the full message */
AF_API int af_device_count(int *count);
AF_API const char *af_version(void);
/* Number of kernels this library has launched since af_init (bench.py's gpu_launches). */
AF_API uint64_t af_kernel_launch_count(void);
/* Debugging aid: cycles the fused kernel's warp roles spent waiting on each pipeline barrier since the last
 * call ([role][total, t0 .. t6], roles FFT / mel / VAD / resample).  All zero unless the library
 * was built with `make STATS=1`. */
AF_API int af_debug_pipe_stats(uint64_t out[32]);
/* Debugging aid: the device and the pinned host allocations the library holds right now, in every object it owns
 * (sessions, batches, detectors, rings, af_host_alloc blocks) and in its per-device caches.  Either pointer may be
 * NULL.  Unlike cudaMemGetInfo, this counts nothing of other processes on the same GPU: a leak check. */
AF_API int af_debug_live_allocations(uint64_t *device, uint64_t *pinned);

/* pinned host memory for the host-buffer entry points (optional but much faster) */
AF_API int af_host_alloc(void **ptr, size_t bytes);
AF_API int af_host_free(void *ptr);

/* ---- AudioFrame::to_mono  (src-tauri/src/modules/audio/capture.rs:30-42) ---------------- */
/* host buffers; out needs ceil(n_samples / channels) floats.  channels == 1 -> copy. */
AF_API int af_to_mono(const float *samples, size_t n_samples, uint16_t channels, float *out, size_t out_cap,
                      size_t *n_out);

/* ---- AudioResampler  (src-tauri/src/modules/audio/resampler.rs:12-112, 169-178) -------- */
typedef struct af_resampler af_resampler;
/* AudioResampler::new (resampler.rs:32-57); create_48k_to_16k (:60-62) == create(48000,16000) */
AF_API int af_resampler_create(uint32_t input_rate, uint32_t output_rate, af_resampler **out);
AF_API void af_resampler_destroy(af_resampler *r);
/* AudioResampler::process (resampler.rs:71-93): equal rates -> copy; otherwise ONE rubato
 * FastFixedIn step: consumes exactly 128 frames (extra ignored), fewer than 128 ->
 * AF_ERR_RESAMPLING_FAILED.  Host buffers. */
AF_API int af_resampler_process(af_resampler *r, const float *input, size_t n, float *out, size_t out_cap,
                                size_t *n_out);
AF_API uint32_t af_resampler_input_rate(const af_resampler *r);   /* resampler.rs:96-98  */
AF_API uint32_t af_resampler_output_rate(const af_resampler *r);  /* resampler.rs:101-103 */
AF_API int af_resampler_needs_resampling(const af_resampler *r);  /* resampler.rs:106-108 */
AF_API size_t af_resampler_chunk_size(const af_resampler *r);     /* 128, or 0 for passthrough */
/* upper bound of the number of output frames produced for n_in input frames */
AF_API size_t af_resample_max_output(uint32_t input_rate, uint32_t output_rate, size_t n_in);
/* exact number of output frames of BatchResampler::process(all n_in) + flush() */
AF_API int af_resample_output_len(uint32_t input_rate, uint32_t output_rate, size_t n_in, size_t *n_out);

/* ---- BatchResampler  (src-tauri/src/modules/audio/resampler.rs:115-166) ---------------- */
typedef struct af_batch_resampler af_batch_resampler;
AF_API int af_batch_resampler_create(uint32_t input_rate, uint32_t output_rate, af_batch_resampler **out);
AF_API void af_batch_resampler_destroy(af_batch_resampler *b);
/* BatchResampler::process (:132-147): buffers input, emits the output of every complete
 * 128-frame chunk.  Equal rates: passthrough (the reference would loop forever there). */
AF_API int af_batch_resampler_process(af_batch_resampler *b, const float *input, size_t n, float *out,
                                      size_t out_cap, size_t *n_out);
/* BatchResampler::flush (:150-166): zero-pads the residual to one chunk and processes it. */
AF_API int af_batch_resampler_flush(af_batch_resampler *b, float *out, size_t out_cap, size_t *n_out);

/* ---- VoiceActivityDetector  (src-tauri/src/modules/audio/vad.rs) ---------------------- */
typedef struct af_vad_config {      /* VadConfig, vad.rs:21-32 */
    float threshold_db;
    float smoothing_factor;
    uint64_t silence_timeout_frames;
    uint64_t min_speech_frames;
} af_vad_config;

enum { AF_VAD_SILENCE = 0, AF_VAD_SPEECH = 1, AF_VAD_ENDING = 2 };   /* VadState, vad.rs:47-54 */

typedef struct af_vad af_vad;
AF_API void af_vad_config_default(af_vad_config *cfg);                 /* vad.rs:34-43 */
AF_API int af_vad_create(const af_vad_config *cfg, af_vad **out);      /* vad.rs:80-88 */
AF_API void af_vad_destroy(af_vad *v);
/* detect (vad.rs:97-154): one frame of any length -> post-transition state */
AF_API int af_vad_detect(af_vad *v, const float *frame, size_t n, uint8_t *state);
/* the same detector driven over many frames [f*hop, f*hop+frame_len) of one host signal in a
 * single launch; writes one state per frame */
AF_API int af_vad_detect_frames(af_vad *v, const float *samples, size_t n, uint32_t frame_len, uint32_t hop,
                                uint8_t *states, size_t states_cap, size_t *n_frames);
AF_API int af_vad_reset(af_vad *v);                                    /* vad.rs:179-184 */
AF_API int af_vad_state(const af_vad *v);                              /* vad.rs:187-189 */
AF_API float af_vad_energy_db(const af_vad *v);                        /* vad.rs:192-194 */
AF_API int af_vad_is_speaking(const af_vad *v);                        /* vad.rs:197-199 */
AF_API uint64_t af_vad_speech_frame_count(const af_vad *v);            /* vad.rs:202-204 */
AF_API float af_vad_smoothed_energy(const af_vad *v);                  /* the field behind energy_db */
/* mean-square frame energy exactly as calculate_energy (vad.rs:157-168), on the GPU */
AF_API int af_vad_frame_energy(const float *frame, size_t n, float *energy);

/* ---- PCM16 wire encode  (src-tauri/src/modules/network/websocket.rs:246-251) ---------- */
AF_API int af_pcm16_encode(const float *samples, size_t n, int16_t *out);
/* The wire payload itself: base64 (standard alphabet, '=' padding) of the little-endian PCM16 bytes -- the
 * "audio_base_64" field of WebSocketClient::send_audio / MessageBuilder::audio_message (websocket.rs:244-254, :338-348).
 * Writes af_pcm16_base64_len(n) = 4 * ceil(2 n / 3) characters (no terminator) into out[out_cap]. */
AF_API size_t af_pcm16_base64_len(size_t n_samples);
AF_API int af_pcm16_base64(const float *samples, size_t n, char *out, size_t out_cap, size_t *n_out);

/* ======================================================================================= */
/* Batched fast path: many independent streams through                                     */
/*   to_mono -> BatchResampler(all)+flush -> STFT/log-mel -> framed VAD                     */
/* in one launch sequence.  Results are identical to driving the per-object API above      */
/* stream by stream.                                                                       */
/* ======================================================================================= */
enum { AF_FMT_F32 = 0, AF_FMT_I16 = 1 };            /* sample format; i16 decodes as s / 32768 */
enum { AF_MEM_DEVICE = 0, AF_MEM_HOST = 1 };        /* where stream data and outputs live */

typedef struct af_pipeline_config {
    uint32_t n_mels;          /* 0 = no STFT/log-mel; else 1..128 (80 and 128 are the BASELINE configs) */
    float f_min, f_max;       /* mel band edges in Hz (0, 8000) */
    float log_floor;          /* log(max(mel, floor)), 1e-10 */
    uint32_t log10;           /* 0 natural log, 1 log10 */
    uint32_t vad_enable;      /* run the VAD */
    af_vad_config vad;
    uint32_t vad_frame_len;   /* 0 -> the STFT frames (400 / 160); else e.g. 320 / 320 (20 ms) */
    uint32_t vad_hop;
    uint32_t write_pcm;       /* write the resampled 16 kHz PCM */
    uint32_t pcm16;           /* batch runs: deliver the PCM as i16 wire samples, (x.clamp(-1,1) * 32767) as i16
                               * (websocket.rs:246-251): af_outputs.pcm then points at int16_t rows and pcm_stride counts
                               * int16_t elements (still a multiple of 4).  Halves the PCM bytes that leave the GPU. */
} af_pipeline_config;

AF_API void af_pipeline_config_default(af_pipeline_config *cfg);

typedef struct af_stream_desc {
    const void *data;         /* interleaved samples [frame][channel] */
    uint64_t n_samples;       /* TOTAL interleaved sample count (AudioFrame::samples.len()) */
    uint32_t sample_rate;     /* AudioFrame::sample_rate; output is always 16 kHz */
    uint16_t channels;        /* AudioFrame::channels */
    uint16_t format;          /* AF_FMT_* */
} af_stream_desc;

typedef struct af_vad_final {   /* detector state after the last frame of a stream */
    float smoothed_energy;
    int32_t state;
    uint64_t silence_frames;
    uint64_t speech_frames;
} af_vad_final;

typedef struct af_outputs {
    float *pcm;               /* [n_streams][pcm_stride]    resampled mono 16 kHz (or NULL); device pointers must be
                               * 16-byte aligned (vector stores), else AF_ERR_INVALID */
    uint64_t pcm_stride;      /* floats per row, multiple of 4 */
    float *logmel;            /* [n_streams][logmel_stride] rows of [frame][mel] (or NULL) */
    uint64_t logmel_stride;   /* floats per row, multiple of 4 */
    uint8_t *vad;             /* [n_streams][vad_stride]    VadState per frame (or NULL) */
    uint64_t vad_stride;
    float *energy;            /* [n_streams][energy_stride] mean-square energy per VAD frame (or NULL) */
    uint64_t energy_stride;
    af_vad_final *vad_final;  /* [n_streams] (or NULL) */
} af_outputs;

typedef struct af_pipeline af_pipeline;
typedef struct af_batch af_batch;

AF_API int af_pipeline_create(const af_pipeline_config *cfg, af_pipeline **out);
AF_API void af_pipeline_destroy(af_pipeline *p);

/* Plans a batch: validates the descriptors, computes per-stream output lengths with the exact
 * chunk recurrence of the reference resampler, builds the device-side stream/tile tables.
 * mem = AF_MEM_DEVICE: desc.data are device pointers (16-byte aligned), the batch can be run
 * many times.  mem = AF_MEM_HOST: desc.data are host pointers, used by af_batch_run_host. */
AF_API int af_batch_create(af_pipeline *p, const af_stream_desc *streams, size_t n_streams, int mem,
                           af_batch **out);
AF_API void af_batch_destroy(af_batch *b);
AF_API size_t af_batch_n_streams(const af_batch *b);
/* per-stream counts (host arrays of n_streams): resampled length, STFT frames, VAD frames */
AF_API int af_batch_counts(const af_batch *b, uint32_t *n_out, uint32_t *n_feat_frames, uint32_t *n_vad_frames);
/* minimal strides (already rounded to the required multiples) */
AF_API int af_batch_strides(const af_batch *b, uint64_t *pcm_stride, uint64_t *logmel_stride,
                            uint64_t *vad_stride);

/* Device-resident run: outputs are device pointers.  Enqueues on `cuda_stream`
 * (a cudaStream_t passed as void*, NULL = the library's own stream) and returns without
 * synchronising when cuda_stream != NULL.  The library's own stream is non-blocking: with cuda_stream == NULL the
 * caller must have finished (synchronised) whatever produced the inputs or still touches the output buffers on
 * other streams, the legacy default stream included. */
AF_API int af_batch_run(af_batch *b, const af_outputs *out, void *cuda_stream);
/* Host-buffer run (the reference-facing call): copies the streams H2D (chunked, overlapped
 * with compute), runs the pipeline and copies the requested outputs back; blocking. */
AF_API int af_batch_run_host(af_batch *b, const af_outputs *out);
/* Per-stream VAD configurations (VoiceActivityDetector::new(config) per caller, vad.rs:21-43, 80-88).  A stream's
 * configuration is the af_vad_config its frames are decided under; by default the pipeline's af_pipeline_config::vad.
 * cfgs holds one configuration per stream (af_batch_n_streams); cfgs == NULL restores the pipeline's for every stream.
 * The configurations apply from the next af_batch_run / af_batch_run_host.  Stream k's states, energies and vad_final
 * are bit for bit those of a one-stream batch whose pipeline has vad = cfgs[k]; PCM and log-mel do not change.  Values
 * are accepted exactly as af_vad_create accepts them (a NaN threshold never detects speech; a smoothing factor outside
 * [0, 1] is scanned sequentially).  A stream whose configuration needs the sequential scan does not move the others off
 * the parallel one: such a batch enqueues one more kernel.  AF_ERR_INVALID when the pipeline has vad_enable == 0.
 * Sharded batches: af_sharded_batch_local(b, r) is an ordinary batch; give each local rank the slice of its streams. */
AF_API int af_batch_set_vad_configs(af_batch *b, const af_vad_config *cfgs);
/* Resampling filter of a batch.  AF_RESAMPLE_CUBIC (the default) is the reference's rubato FastFixedIn cubic, which has
 * no anti-alias filter: everything between 8 kHz and the input's Nyquist folds into the 0-8 kHz band.
 * AF_RESAMPLE_POLYPHASE is scipy.signal.resample_poly(m, q, p)'s default filter on the downmix m, for R / 16000 = p / q
 * reduced and L = 10 max(p, q): h = firwin(2L + 1, 1 / max(p, q), window=('kaiser', 5.0)) in f64, cast to f32, times
 * (float)q; y[n] = sum_k m[k] h[n p + L - k q] over ascending k (m = 0 outside the stream) as a chain of fmaf from
 * +0.0f; 16 kHz streams are copied.  Passband within 0.02 dB to 6 kHz, at most -56.8 dB from 10 kHz up (for every rate
 * above 16 kHz), -6 dB at 8 kHz.  Counts and strides do not change (n_out stays the cubic path's), and everything
 * downstream (PCM rows, pcm16, log-mel, energies, VAD) is what the batch computes for 16 kHz mono f32 streams holding
 * y[0 .. n_out).  Every stream's rate must reduce to max(p, q) <= 65536 (every common capture rate does), else
 * AF_ERR_RESAMPLING_FAILED naming the first stream that does not; AF_ERR_INVALID for a null batch or an unknown
 * filter.  On an error nothing changes.  The filter applies from the next af_batch_run / af_batch_run_host.
 * AF_RESAMPLE_CUBIC frees what the polyphase filter allocated (a 16 kHz row block, tap tables and tile tables).
 * Sharded batches: set it on af_sharded_batch_local(b, r) for each local rank. */
enum { AF_RESAMPLE_CUBIC = 0, AF_RESAMPLE_POLYPHASE = 1 };
AF_API int af_batch_set_resampler(af_batch *b, uint32_t filter);
/* The polyphase taps for input_rate -> output_rate (host only, no GPU needed): returns 2L + 1 and writes the first cap
 * taps to h and the reduced ratio to *p, *q (any may be NULL); 0 when max(p, q) > 65536. */
AF_API size_t af_debug_polyphase_filter(uint32_t input_rate, uint32_t output_rate, float *h, size_t cap, uint32_t *p, uint32_t *q);
/* One-shot convenience: create + run_host + destroy. */
AF_API int af_pipeline_run(af_pipeline *p, const af_stream_desc *streams, size_t n_streams,
                           const af_outputs *out);

/* which variant of the fused kernel to launch (default "auto"); for tests and ncu comparisons.
 * names: "auto", "sync" (plain loads), "tma" (bulk-copy staged input).  Returns AF_ERR_INVALID
 * for unknown names. */
AF_API int af_set_kernel_variant(const char *name);

/* ---- VAD segmentation (consumer of VadState; SURVEY 8(f) f1) --------------------------- */
/* device buffers: states [n_streams][vad_stride] -> seg [n_streams][seg_cap][2] = [start,end)
 * frames, n_seg [n_streams].  A segment runs from the first Speech frame to the frame that
 * reports Ending (inclusive) or that falls back to Silence (exclusive). */
AF_API int af_vad_segments(const uint8_t *states, uint64_t vad_stride, const uint32_t *n_frames,
                           size_t n_streams, uint32_t *seg, uint32_t seg_cap, uint32_t *n_seg,
                           void *cuda_stream);
/* Pre-roll, in place on af_vad_segments' output (device pointers; the first min(n_seg, seg_cap)
 * segments of each stream): segment k [start, end) becomes [max(start - P, end of segment k - 1,
 * 0), end), the first segment's predecessor ending at 0.  The segments stay disjoint and in
 * order, and af_vad_gate then keeps the P frames before every onset (fewer where the previous
 * segment or the stream's start is closer).  Any P; P = 0 leaves seg untouched. */
AF_API int af_vad_segments_preroll(uint32_t *seg, uint32_t seg_cap, const uint32_t *n_seg, size_t n_streams,
                                   uint32_t preroll_frames, void *cuda_stream);

/* ---- VAD-gated output (SURVEY 8(f) f1, second half) ------------------------------------- */
/* What the reference's spec wants in front of the wire (specs/0001-spec.md:466: drop the silent stretches before
 * ScribeClient::send_audio, src-tauri/src/modules/network/scribe_client.rs:194-196): only the audio and the feature
 * rows of the speech segments, packed.  Frame f of a segment [start, end) contributes its hop -- samples
 * [f*hop, (f+1)*hop) of the 16 kHz row -- and log-mel row f; the kept frames of a stream are stored back to back in
 * order.  seg_offset[s][k] is the compacted frame index where segment k starts (PCM offset = that times hop),
 * seg_offset[s][n_seg] == n_frames[s] is the number of kept frames.  All pointers are device pointers;
 * seg / n_seg are af_vad_segments' outputs (segments beyond seg_cap are ignored). */
typedef struct af_gate_outputs {
    float *pcm;               /* [n_streams][pcm_stride]    gated 16 kHz samples (or NULL) */
    uint64_t pcm_stride;
    float *logmel;            /* [n_streams][logmel_stride] gated rows of [frame][mel] (or NULL) */
    uint64_t logmel_stride;
    uint32_t *seg_offset;     /* [n_streams][seg_cap + 1] */
    uint32_t *n_frames;       /* [n_streams] kept frames */
} af_gate_outputs;
AF_API int af_vad_gate(const float *pcm, uint64_t pcm_stride, const float *logmel, uint64_t logmel_stride, uint32_t n_mels,
                       const uint32_t *n_out, uint32_t hop, const uint32_t *seg, uint32_t seg_cap, const uint32_t *n_seg,
                       size_t n_streams, const af_gate_outputs *out, void *cuda_stream);

/* ======================================================================================= */
/* Multi-GPU: independent streams sharded over the GPUs of one box, results gathered with NCCL  */
/* (SURVEY 8(e)).  Streams never talk to each other, so the data path has NO collective; the only */
/* exchange is the gather of the per-stream VAD states to every GPU, issued on a side stream so    */
/* that the next batch never waits for it.  Two ways to form the communicator:                     */
/*   - af_init_multi(n): ONE process (e.g. the Rust host) drives GPUs 0..n-1 (ncclCommInitAll);    */
/*   - one process per GPU: af_init(local_gpu), rank 0 calls af_comm_unique_id, the host ships the  */
/*     128 bytes to the other ranks by any channel, every rank calls af_comm_init_rank.             */
/* NCCL is loaded at run time (libnccl.so.2); single-GPU use never touches it.                      */
/* ======================================================================================= */
AF_API int af_init_multi(int n_gpus);
AF_API int af_comm_unique_id(uint8_t id[128]);
AF_API int af_comm_init_rank(int n_ranks, int rank, const uint8_t id[128]);
AF_API int af_comm_size(void);                  /* ranks of the communicator, 0 when there is none */
AF_API int af_comm_shutdown(void);
/* Contiguous blocks of stream indices, balanced by input BYTES (44.1 kHz and 48 kHz streams differ by 8 %):
 * shard r owns streams [first[r], first[r + 1]); first has n_shards + 1 entries.  Pure host code. */
AF_API int af_shard_partition(const af_stream_desc *streams, size_t n_streams, int n_shards, size_t *first);

typedef struct af_sharded_batch af_sharded_batch;
typedef struct af_sharded_outputs {             /* per rank; only the entries of this process's ranks are read */
    af_outputs shard[AF_MAX_GPUS];              /* device pointers on the rank's GPU, rows = the rank's streams */
} af_sharded_outputs;
/* Plans n_streams GLOBAL streams over the communicator's ranks (af_shard_partition) and builds the batches of the
 * ranks this process owns (all of them after af_init_multi, one after af_comm_init_rank).  Every process passes the
 * same descriptor list; the `data` of streams owned elsewhere is not used (may be NULL).  mem as in af_batch_create;
 * AF_MEM_DEVICE data must live on the owner's GPU. */
AF_API int af_sharded_batch_create(af_pipeline *p, const af_stream_desc *streams, size_t n_streams, int mem,
                                   af_sharded_batch **out);
AF_API void af_sharded_batch_destroy(af_sharded_batch *b);
/* rank r owns streams [*first, *first + *count); *device = its GPU when this process owns the rank, else -1 */
AF_API int af_sharded_batch_shard(const af_sharded_batch *b, int rank, size_t *first, size_t *count, int *device);
AF_API af_batch *af_sharded_batch_local(af_sharded_batch *b, int rank);   /* the rank's ordinary batch (counts, strides); NULL if remote */
/* Runs every local shard on its GPU (all GPUs concurrently, nothing blocks in between).  gather != 0: the VAD kernel
 * of each shard writes its states straight into the rank's slot of a double-buffered gather buffer and ONE in-place
 * ncclAllGather per GPU follows on the side stream; shard[r].vad is then ignored.  async == 0: returns when every GPU
 * (and the gather) is done; else af_sharded_batch_wait does that. */
AF_API int af_sharded_batch_run(af_sharded_batch *b, const af_sharded_outputs *out, int gather, int async);
AF_API int af_sharded_batch_wait(af_sharded_batch *b);
/* Orders the compute stream of every local GPU after the last gather WITHOUT blocking the host: work (or an event)
 * enqueued afterwards sees the gathered states. */
AF_API int af_sharded_batch_join(af_sharded_batch *b);
/* The gathered states of the LAST run on a local rank's GPU: row (r * rows_per_rank + i) holds stream i of rank r,
 * n_vad_frames[global stream] of them valid (host array of n_streams, may be NULL).  The buffer is reused by the run
 * after the next one. */
AF_API int af_sharded_batch_gathered(af_sharded_batch *b, int rank, const uint8_t **states, uint64_t *row_stride,
                                     uint64_t *rows_per_rank, uint32_t *n_vad_frames);
/* The same result on the host, in GLOBAL stream order: states[n_streams][stride] (stride >= the longest stream's
 * frame count).  Waits for the gather. */
AF_API int af_sharded_batch_gathered_host(af_sharded_batch *b, int rank, uint8_t *states, uint64_t stride);
/* Device time of the last gather on a local rank (side stream, event to event), milliseconds. */
AF_API int af_sharded_batch_gather_ms(af_sharded_batch *b, int rank, float *ms);
/* Host-buffer form (mem == AF_MEM_HOST): `out` holds rows for ALL n_streams streams in host memory; every local shard
 * runs af_batch_run_host on its GPU from its own host thread, writing its rows.  Blocking. */
AF_API int af_sharded_batch_run_host(af_sharded_batch *b, const af_outputs *out);

/* ---- host-side planning diagnostics (no GPU needed; used by the CPU test-suite) ---------- */
/* smallest f32 energy e with 20*log10f(e) > threshold_db under the host libm (NaN if none):
 * the device compares energies against this instead of taking a log (DESIGN.md, VAD). */
AF_API float af_debug_vad_energy_threshold(float threshold_db);
/* the f32 fractional offsets the host plan derives for the first n_chunks 128-frame chunks of
 * an (input_rate -> output_rate) stream; returns the number of outputs (may exceed cap). */
AF_API size_t af_debug_resample_plan(uint32_t input_rate, uint32_t output_rate, size_t n_chunks, float *frac,
                                     size_t cap, int *mode);
/* the order in which a batch launches its tiles over n_ctas CTAs (CTA c runs positions c, c + n_ctas, ...), given
 * each tile's step count: order[i] = tile placed at position i (n entries).  Returns the step count of the busiest CTA. */
AF_API uint64_t af_debug_tile_order(const uint32_t *steps, size_t n, uint32_t n_ctas, uint32_t *order);

/* ---- streaming sessions (persistent per-stream state; BASELINE config 5) ---------------- */
typedef struct af_session af_session;
/* n_streams concurrent streams of one (rate, channels, format); state (resampler position,
 * residual input, STFT overlap, VAD) stays on the device between ticks. */
AF_API int af_session_create(af_pipeline *p, size_t n_streams, uint32_t sample_rate, uint16_t channels,
                             uint16_t format, uint32_t max_tick_samples, af_session **out);
AF_API void af_session_destroy(af_session *s);
/* One tick: every stream pushes `n_samples` interleaved samples (device or host per `mem`,
 * rows `in_stride` samples apart).  Outputs produced by this tick are appended at the row
 * starts of `out`; counts (host arrays of n_streams, may be NULL) receive how many
 * PCM samples / feature frames / VAD frames each stream emitted.  With the VAD on, out->vad_final
 * (if set) receives every stream's detector state after its last frame so far on every push of any
 * kind, a push that completes no frame included. */
AF_API int af_session_push(af_session *s, const void *data, uint64_t in_stride, uint32_t n_samples, int mem,
                           const af_outputs *out, uint32_t *n_pcm, uint32_t *n_feat, uint32_t *n_vad);
AF_API int af_session_reset(af_session *s);

/* ---- level metering for the UI events ---------------------------------------------------- */
/* AudioLevel{level, peak} (src-tauri/src/events/mod.rs:41,73-75) and VolumeLevel{level, is_speech}
 * (src-tauri/src/modules/events/mod.rs:22,182-185) as by-products of a session tick.  The reference only declares
 * the payloads; the values are defined here: level_db = VoiceActivityDetector::energy_db() (vad.rs:192-194:
 * 20*log10 of the smoothed energy after the tick's last frame, -inf when it is <= 0 or the VAD is off),
 * peak = max |y| over the 16 kHz samples the tick produced (0 if none), is_speech = is_speaking() (vad.rs:197-199).
 * Enable once, then read after every push; host arrays of n_streams, any may be NULL. */
AF_API int af_session_enable_levels(af_session *s, int enable);
AF_API int af_session_levels(const af_session *s, float *level_db, float *peak, uint8_t *is_speech);

/* ---- streaming wire output: what WebSocketClient::send_audio sends, per tick (websocket.rs:244-254) ----------------
 * With the wire output enabled, every push (af_session_push, af_session_push_rings) leaves one payload per stream:
 *   gate = 0: every 16 kHz sample the tick produced (the n_pcm samples af_session_push returns as f32);
 *   gate = 1: only the speech (specs/0001-spec.md:466, scribe_client.rs:194-196; needs vad_enable and a VAD hop no
 *             longer than its frame): for every VAD frame f completed in this tick that lies in a segment of
 *             af_vad_segments -- a Speech frame, or the Ending frame that closes one -- the frame's hop, samples
 *             [f*hop, (f+1)*hop) of the stream's 16 kHz signal, kept frames in order.  Concatenating the gated payloads
 *             of all ticks gives af_vad_gate's PCM over the concatenated session PCM and states.  A frame completes
 *             frame_len - hop samples after its hop ends, so the gated payload trails the newest samples by at least
 *             that overlap (240 samples = 15 ms with the STFT frames, none with the 20 ms frames of
 *             vad_frame_len = vad_hop = 320), plus the samples of a frame not yet complete.
 * Encoding: PCM16 = (x.clamp(-1,1) * 32767) as i16, NaN -> 0 (websocket.rs:246-251); base64 = standard alphabet with '='
 * padding over the little-endian bytes of THIS tick's payload alone (one send_audio call per tick), no terminator,
 * af_pcm16_base64_len(n_samples) characters.  An empty payload has 0 samples and 0 characters.
 * Per stream and tick an af_wire_tick (the event fields are 0 without the VAD):
 *   started   segments whose first frame (a Speech frame whose predecessor, across ticks, is not Speech) is in the tick;
 *   ended     segments closed by a frame of the tick: an Ending frame, or a Silence frame after a Speech frame;
 *   in_speech the stream's latest completed frame is Speech (the tick's last frame; an earlier one if it completed none);
 *   continued gated only: payload samples at the front that belong to the segment already open when the tick began
 *             (the rest belongs to segments started in the tick); 0 ungated, where payloads are not frame-aligned.
 * first_frame is the global index of the tick's first completed frame (the same for all streams in lockstep; stream 0's
 * once streams have their own timelines, see af_session_wire_first_frames).
 * af_session_reset clears the carried segment state. */
typedef struct af_wire_config {
    uint32_t gate;            /* 0: every 16 kHz sample of the tick; 1: only the hops of its segment frames (needs the VAD) */
    uint32_t pcm16;           /* produce the PCM16 samples */
    uint32_t base64;          /* produce the base64 text of their little-endian bytes (no terminator) */
    int32_t mem;              /* AF_MEM_HOST: session-owned pinned host rows; AF_MEM_DEVICE: device rows on the session's GPU */
} af_wire_config;
typedef struct af_wire_tick {
    uint32_t n_samples, n_chars, continued;
    uint16_t started, ended;
    uint8_t in_speech, pad[3];
} af_wire_tick;
/* cfg NULL: off.  AF_ERR_INVALID for gate = 1 without the VAD (or with vad_hop > vad_frame_len), neither pcm16 nor
 * base64, or a bad mem.  Allocates the rows: a tick's payload is bounded when the session is created. */
AF_API int af_session_enable_wire(af_session *s, const af_wire_config *cfg);
/* The payloads of the last push: row k of pcm16 (int16 elements, stride in elements) and of base64 (bytes) holds stream
 * k's payload; rows are NULL (stride 0) for an encoding that is off, and stay valid until the next push.  ticks: host
 * array of n_streams (may be NULL).  AF_ERR_INVALID before the first push since af_session_enable_wire. */
AF_API int af_session_wire(const af_session *s, const int16_t **pcm16, uint64_t *pcm16_stride, const char **base64,
                           uint64_t *base64_stride, af_wire_tick *ticks, uint64_t *first_frame);
/* ---- wire features: the speech-gated log-mel rows beside the gated PCM (SURVEY 8(f) f1 on a session) ----------------
 * With the gated wire output on (gate = 1) and its features enabled, every push also leaves, per stream, the log-mel row
 * of every frame the gated payload keeps in this tick -- a Speech frame in a segment, or the Ending frame that closes
 * one -- in order, n_mels floats each, back to back.  For every stream k and tick: n_frames[k] * hop == the
 * af_wire_tick's n_samples; the rows are, bit for bit, the kept frames' rows of the tick's log-mel (what out->logmel
 * receives; the tick computes it whether or not out->logmel is set); the segment open when the tick began owns the first
 * continued / hop rows; and concatenated over every tick since the stream's start they are af_vad_gate's log-mel over the
 * concatenated session log-mel and states.  Log-mel row f belongs to VAD frame f, so the VAD must run on the STFT frames
 * (vad_frame_len 0, or 400 / 160), as for af_vad_gate.  Everything the gated payload defines holds for the rows: ends
 * close segments, af_session_reset_streams / af_session_restart_streams drop an open one, an imported stream continues
 * its open segment, per-stream VAD configurations decide the frames.  A stream record carries nothing more.
 * enable != 0: mem AF_MEM_HOST (session-owned pinned rows) or AF_MEM_DEVICE (rows on the session's GPU); the rows are
 * sized here for the session's bound of frames per tick.  AF_ERR_INVALID, and nothing changes, when the wire output is
 * off or ungated, for n_mels == 0 or vad_enable == 0, VAD frames other than the STFT frames, or a bad mem.  enable == 0:
 * off.  Every af_session_enable_wire call (off, or a new configuration) turns the features off as well. */
AF_API int af_session_enable_wire_features(af_session *s, int enable, int mem);
/* The rows of the last push: row k (stride floats apart, a multiple of 4) holds stream k's n_frames[k] * n_mels floats,
 * valid until the next push.  n_frames: host array of n_streams (may be NULL).  AF_ERR_INVALID whenever af_session_wire
 * is (before the first push since enabling, after an import, after a failed push) and while the features are off. */
AF_API int af_session_wire_features(const af_session *s, const float **rows, uint64_t *stride, uint32_t *n_frames);
/* ---- wire pre-roll: every speech segment of the gated payload reaches back P frames ------------------------------------
 * The detector says Speech a few frames after an onset (the smoothed energy has to cross the threshold), and a quiet
 * lead-in below the threshold never does; a gated payload that starts at the detected frame clips the first phoneme.
 * With a pre-roll of P frames, a segment start g (a kept frame that is Speech after a frame that is not, across ticks)
 * also brings in its pre-roll frames [max(g - P, k + 1, o), g): k is the last kept frame before g (-1 if none), so the
 * pre-roll never reaches into the previous segment or repeats a frame; o is the stream's origin, the first frame after
 * its start (creation, af_session_reset, af_session_reset_streams, af_session_restart_streams, the push after an end),
 * after an import into its slot, or after the latest af_session_set_wire_preroll call.  A tick's gated payload then
 * holds, in frame order, every kept frame completed in the tick and every pre-roll frame of a segment started in it,
 * whichever push completed that frame.  Per stream and tick: n_frames * hop == n_samples; the PCM16 and base64 rows
 * encode those frames' hops (the base64 this tick's bytes alone); the wire features, when on, are the log-mel rows of
 * the same frames; concatenated since the origin, the payloads are af_vad_gate's output over the stream's PCM, log-mel
 * and states since the origin with the segments of af_vad_segments_preroll.  started, ended, in_speech and continued
 * are those without the pre-roll: the pre-roll belongs to its new segment, after the continued samples, and only
 * n_samples and n_chars grow.  The history of up to P frames stays on the session's GPU; a stream record does not carry
 * it (the record's layout depends on the framing alone), so an import starts a new origin.
 * frames: 0 to AF_WIRE_PREROLL_MAX.  Grows the wire rows by frames * hop samples and the feature rows by
 * frames * n_mels floats, allocates the history for `frames`, and makes the next push every stream's origin; the last
 * push's rows are released (af_session_wire refuses until the next push).  frames = 0 frees the history: the session
 * then runs as one that never set a pre-roll.  AF_ERR_INVALID, and nothing changes, when the gated wire output is off or
 * for frames > AF_WIRE_PREROLL_MAX.  Every af_session_enable_wire and af_session_enable_wire_features call sets the
 * pre-roll back to 0: set it last. */
#define AF_WIRE_PREROLL_MAX 100
AF_API int af_session_set_wire_preroll(af_session *s, uint32_t frames);
/* ---- wire segments: where each utterance lies in a tick's gated payload -------------------------------------------------
 * A coarse or ragged tick (1 s ticks, af_session_push_rings_available after a stall) can hold several utterances back to
 * back, and with a pre-roll a payload reaches back into earlier pushes; the counts of af_wire_tick cannot cut it apart
 * or timestamp it.  With the gated wire on and its segment table enabled, every push also leaves a list of pieces per
 * stream.  A piece is the part of one segment that lies in this tick's payload; segments are those of af_vad_segments,
 * pre-rolled as af_session_set_wire_preroll defines.  Pieces are listed in payload order.  Per stream and tick:
 *   - pieces tile the payload: the first starts at offset 0, offset[i + 1] == offset[i] + n_frames[i], and
 *     sum(n_frames) * hop == n_samples;
 *   - pieces without AF_WIRE_SEG_CONTINUED number `started`, pieces with AF_WIRE_SEG_CLOSED number `ended`; a CONTINUED
 *     piece comes first, and its n_frames * hop == continued;
 *   - every piece but the last is CLOSED; the last lacks CLOSED exactly when in_speech is 1.  A tick that completes no
 *     frame and closes nothing has no pieces, even while a segment is open;
 *   - closing-only piece: a segment open when the tick began that closes with no payload frame in the tick (the tick's
 *     first frame is Silence after Speech, or an end comes with no completed frame) is one piece with
 *     CONTINUED | CLOSED and n_frames = 0, frame = 0.  No other piece has 0 frames;
 *   - a reset or restart drops an open segment (the next tick has no CONTINUED piece); after an import, a segment open
 *     in the record continues with a CONTINUED piece; under a pre-roll an import is an origin, as for the payload.
 * Concatenated since the stream's origin, each CONTINUED piece joined to the open segment and frames made global as
 * first_frames[k] + frame (af_session_wire_first_frames), the pieces are exactly af_vad_segments (+
 * af_vad_segments_preroll with the session's P) over the stream's concatenated states, and their cumulative payload
 * offsets are af_vad_gate's seg_offset.  The table counts VAD frames, so it needs no STFT frames (20 ms VAD frames
 * work).  Payload sample offset * hop and wire-feature row `offset` are the piece's first. */
#define AF_WIRE_SEG_CONTINUED 1   /* belongs to the segment open when the tick began */
#define AF_WIRE_SEG_CLOSED 2      /* the segment closes in this tick: its Ending frame, a Silence frame after Speech, or the end */
typedef struct af_wire_segment {
    int32_t frame;            /* the piece's first payload frame, relative to the tick's first completed frame
                                 (af_session_wire_first_frames[k]); negative when a pre-roll reaches into earlier pushes */
    uint32_t offset;          /* payload frame index where the piece starts: sample offset * hop, wire-feature row offset */
    uint32_t n_frames;        /* payload frames of the piece (0 only for the closing-only piece) */
    uint16_t preroll;         /* pre-roll frames at the piece's front: the detected onset is frame + preroll (0 if CONTINUED) */
    uint8_t flags;            /* AF_WIRE_SEG_CONTINUED | AF_WIRE_SEG_CLOSED */
    uint8_t pad;              /* 0 */
} af_wire_segment;            /* 16 bytes */
/* enable != 0: mem AF_MEM_HOST (session-owned pinned rows) or AF_MEM_DEVICE (rows on the session's GPU), sized for the
 * session's bound of frames per tick T: a tick has at most started + 1 pieces and started <= ceil(T / 2), so a row holds
 * ceil(T / 2) + 1 entries.  enable == 0: off, the rows are freed.  AF_ERR_INVALID, and nothing changes, when the wire
 * output is off or ungated, or for a bad mem.  Neither the features nor the pre-roll change: unlike the other enable
 * calls this one does NOT set the pre-roll back to 0 (a row's size does not depend on it).  Every af_session_enable_wire
 * call turns the table off. */
AF_API int af_session_enable_wire_segments(af_session *s, int enable, int mem);
/* The table of the last push: row k (stride entries apart) holds stream k's n_segs[k] pieces, valid until the next
 * push.  n_segs: host array of n_streams (may be NULL).  AF_ERR_INVALID whenever af_session_wire is (before the first
 * push since enabling, after an import, after a failed push) and while the table is off. */
AF_API int af_session_wire_segments(const af_session *s, const af_wire_segment **rows, uint64_t *stride, uint32_t *n_segs);

/* ---- RingBuffer  (src-tauri/src/modules/audio/capture.rs:84-161): capture hand-off ------ */
/* The cpal callback writes captured f32 samples, the processing task reads them.  Same semantics as the
 * reference: one slot stays free (capacity - 1 usable), a write drops what does not fit and returns the
 * count written, a read returns min(size, available).  The storage is pinned host memory when a device is
 * bound, so a session tick copies straight out of it.  Calls lock like the reference's Mutex<Vec<f32>>. */
typedef struct af_ring af_ring;
#define AF_RING_EMPTY (-1) /* af_ring_read: nothing available -- the reference's `None`, not an error */
AF_API int af_ring_create(size_t capacity_samples, af_ring **out);       /* RingBuffer::new  capture.rs:91-99 */
AF_API void af_ring_destroy(af_ring *r);
AF_API size_t af_ring_capacity(const af_ring *r);
AF_API size_t af_ring_write(af_ring *r, const float *data, size_t n);    /* RingBuffer::write capture.rs:101-121 */
AF_API int af_ring_read(af_ring *r, float *out, size_t size, size_t *n_read);   /* RingBuffer::read capture.rs:123-147 */
AF_API size_t af_ring_available(const af_ring *r);                       /* capture.rs:149-154 */
AF_API void af_ring_clear(af_ring *r);                                   /* capture.rs:156-161 */
/* AudioCapturer::read_frame (capture.rs:310-319) for every stream of a session at once: takes exactly
 * n_samples from each of the n_streams rings and pushes them as one tick (af_session_push).  Nothing is
 * consumed unless every ring holds n_samples. */
AF_API int af_session_push_rings(af_session *s, af_ring *const *rings, uint32_t n_samples, const af_outputs *out,
                                 uint32_t *n_pcm, uint32_t *n_feat, uint32_t *n_vad);

/* ---- independent stream timelines: ragged ticks, end of stream, per-stream restart ----------------------------------
 * Every stream of a session has its own timeline: stream k of a session behaves exactly like a one-stream session pushed
 * the same ticks -- per tick the output of BatchResampler::process (resampler.rs:132-147) on that stream's samples, the
 * frames they complete, the VAD over those frames, the wire payload and record of those frames, its levels.  af_session_push
 * on a session whose streams have diverged is af_session_push_streams with all counts equal and no end; af_session_reset
 * returns every stream to the common start.  All argument errors (a count above max_tick_samples: AF_ERR_CAPACITY; a
 * partial frame, in_stride below a count, a stream index out of range, a null array: AF_ERR_INVALID; an output row too
 * short for the largest count: AF_ERR_CAPACITY) are reported before any state changes.  After AF_ERR_CUDA, reset.
 *
 * One tick in which stream k pushes n_samples[k] interleaved samples (0 allowed; a whole number of frames; at most
 * max_tick_samples) from the start of row k, rows in_stride samples apart (in_stride >= every n_samples[k]).
 * end (may be NULL): end[k] != 0 ends stream k after this tick's samples -- BatchResampler::flush (resampler.rs:150-166):
 * the residual input is zero-padded to one 128-frame chunk and resampled, every frame completed by it is emitted, the
 * rest of the 16 kHz tail is dropped.  Its next push starts afresh, exactly like a stream of a newly created session.
 * An end closes a wire segment that is still open (as af_vad_segments closes one at the last frame): that tick counts it
 * in `ended` and reports in_speech = 0.
 * Outputs go to row k's start; n_pcm[k] / n_feat[k] / n_vad[k] say how many each stream emitted (rows must hold the
 * largest).  vad_final[k] of an ended stream is its detector after its last frame. */
AF_API int af_session_push_streams(af_session *s, const void *data, uint64_t in_stride, const uint32_t *n_samples,
                                   const uint8_t *end, int mem, const af_outputs *out,
                                   uint32_t *n_pcm, uint32_t *n_feat, uint32_t *n_vad);
/* Streams streams[0..n) start afresh at their next push without a flush: pending input, 16 kHz tail, detector and open
 * wire segment are discarded (the caller went away).  Other streams are untouched.  A stream may be listed twice. */
AF_API int af_session_reset_streams(af_session *s, const uint32_t *streams, size_t n);
/* AudioCapturer::read_frame(max) (capture.rs:310-319, RingBuffer::read returns min(size, available)) for every stream:
 * takes min(max_samples, available) samples from each ring, rounded down to whole frames (an empty ring pushes 0; a
 * partial frame stays in the ring), and pushes them with af_session_push_streams.  Nothing is consumed when an argument
 * is refused; max_samples above max_tick_samples is AF_ERR_CAPACITY. */
AF_API int af_session_push_rings_available(af_session *s, af_ring *const *rings, uint32_t max_samples, const uint8_t *end,
                                           const af_outputs *out, uint32_t *n_pcm, uint32_t *n_feat, uint32_t *n_vad);
/* Per stream (host array of n_streams): the index, in that stream's own frame sequence since its last start, of the
 * first frame completed by the last push.  af_session_wire's first_frame is this value for stream 0.  AF_ERR_INVALID
 * when af_session_wire would be. */
AF_API int af_session_wire_first_frames(const af_session *s, uint64_t *first_frame);

/* ---- sessions of mixed capture formats: each stream with its own rate and channel count ----------------------------
 * Capture devices differ (AudioFrame carries its own sample_rate and channels, capture.rs:30-42; every BatchResampler
 * is built for its own device's rate, resampler.rs:115-166).  A session created with af_session_create_formats admits
 * a list of formats; every stream is in one of them at a time and a restarted stream may take another.  Stream k
 * behaves exactly like a one-stream af_session_create session of its current format pushed the same ticks: PCM,
 * frames, VAD, vad_final, the wire payload and its record, the levels and af_session_wire_first_frames.  The output is
 * 16 kHz for every format.  On every push, n_samples[k] must be a whole number of frames of stream k's channels
 * (AF_ERR_INVALID) and at most its format's max_tick_samples (AF_ERR_CAPACITY); the other rules of af_session_push_streams
 * hold, and all errors are reported before any state changes.  On such a session:
 *   af_session_push                  is af_session_push_streams with all counts equal (the lockstep tick runs only
 *                                    while every stream is in one format at one position);
 *   af_session_push_rings            takes exactly n_samples from every ring, under the same count checks;
 *   af_session_push_rings_available  refuses a max_samples above the largest bound over the formats (AF_ERR_CAPACITY);
 *                                    stream k takes min(max_samples, its format's max_tick_samples, available), rounded
 *                                    down to whole frames of its channels (a single-format session sees no change);
 *   af_session_reset                 returns every stream to the common start in its current format. */
typedef struct af_stream_format {
    uint32_t sample_rate;        /* the stream's capture rate; output is always 16 kHz */
    uint16_t channels;           /* interleaved channels */
    uint16_t pad;                /* 0 */
    uint32_t max_tick_samples;   /* bound of one tick's interleaved samples for a stream in this format */
} af_stream_format;              /* 12 bytes */
/* A session that admits the n_formats formats listed (1 to 65536).  Stream k starts in formats[stream_format[k]]
 * (stream_format NULL: every stream in formats[0]).  sample_format (AF_FMT_F32 / AF_FMT_I16) is the same for the
 * whole session, so in_stride keeps counting samples.  The buffers are sized for the largest bound over the
 * admitted formats.  AF_ERR_INVALID for n_formats == 0, a zero rate, channel count or bound, a nonzero pad, a
 * stream_format index out of range or a bound too large for a session; AF_ERR_RESAMPLING_FAILED for an unsupported
 * ratio.  af_session_create(p, n, rate, channels, fmt, max, out) is this call with the one format
 * {rate, channels, 0, max}. */
AF_API int af_session_create_formats(af_pipeline *p, size_t n_streams, const af_stream_format *formats, size_t n_formats,
                                     const uint32_t *stream_format, uint16_t sample_format, af_session **out);
/* Streams streams[i] start afresh at their next push in formats[format[i]]: af_session_reset_streams plus a new
 * format.  A stream that ended with a flush has nothing left to discard.  A stream or format index out of range is
 * AF_ERR_INVALID, and nothing changes. */
AF_API int af_session_restart_streams(af_session *s, const uint32_t *streams, const uint32_t *format, size_t n);

/* ---- per-stream VAD configurations: every caller's VoiceActivityDetector::new(config) (vad.rs:21-43, 80-88) ----------
 * Stream streams[i] takes the configuration cfgs[i] (a stream listed twice takes its last entry); streams not listed keep
 * theirs, by default the pipeline's af_pipeline_config::vad.  Every frame completed by the next push and later is decided
 * under the new configuration; frames of earlier pushes are not revisited.  The detector keeps its state (smoothed
 * energy, state, silence and speech counters): this is the reference detector with its `config` field replaced between
 * two detect calls.  The reference has no such setter, so this is a definition (DESIGN.md section 10).
 * The configuration belongs to the slot: it survives af_session_reset, af_session_reset_streams,
 * af_session_restart_streams and an end.  A caller who takes over a slot sets it before or after the restart, before
 * the first push, and gets a fresh detector with that configuration, exactly VoiceActivityDetector::new(config).
 * Stream k behaves exactly like a one-stream session whose pipeline has its configuration, pushed the same ticks: states,
 * vad_final, levels, the gated wire payload and its records, af_session_wire_first_frames.  A session whose streams all
 * have the pipeline's configuration runs exactly as one that never called this.  Values are accepted as af_vad_create
 * accepts them.  AF_ERR_INVALID, before anything changes, when the pipeline has vad_enable == 0, for a stream index out of
 * range and for null arrays with n > 0. */
AF_API int af_session_set_vad_configs(af_session *s, const uint32_t *streams, const af_vad_config *cfgs, size_t n);

/* ---- stream records: a live stream leaves its slot and continues in another session, on any GPU ---------------------
 * A stream record is a self-contained byte image of one stream, written by the library: resampler position, input
 * history and residual, the 16 kHz carry of unfinished frames, the detector, the open wire segment and the stream's VAD
 * configuration.  The layout is private; a record is an in-memory hand-off between sessions of the same library build (it
 * carries a version, and a different one is refused), not a storage format.
 * Definition: export stream j of session A after some push and import the record into slot k of session B.  From then on
 * stream k of B behaves exactly like stream j of A would have when pushed the same ticks: PCM, frame counts, VAD states,
 * vad_final, energies, log-mel (bitwise: the same kernels compute it), the wire payload and its af_wire_tick records
 * (`continued` counts into a segment that was open before the move), the levels and af_session_wire_first_frames (which
 * keeps counting in the stream's own frame sequence).  B may differ from A in everything else: number of streams, GPU,
 * list of formats, max_tick_samples bounds, sample type (the state is mono f32), whether its streams have diverged, wire
 * and levels settings, and its pipeline's default vad.
 * Compatibility: B's framing must equal A's -- features or VAD on at all, vad_frame_len / vad_hop as the session uses them,
 * and vad_enable -- and B must admit a format with the record's rate and channel count.  Everything downstream of the
 * framing (n_mels, band edges, log settings, write_pcm) is B's.
 * The VAD configuration travels with the caller: the record holds the stream's effective af_vad_config (its own, else A's
 * pipeline's), and the import gives the slot that configuration exactly as af_session_set_vad_configs would (a slot whose
 * configuration equals B's pipeline's does not count as custom).  This is the one exception to "the configuration belongs
 * to the slot": a caller who takes over a slot by an import brings their own detector.
 * Wire state: with A's wire output on, the record carries the state of the stream's latest completed frame; otherwise the
 * import opens no segment, as af_session_enable_wire does.
 * A stream exported after an end or af_session_reset_streams, or before its first push, is a pending restart in its
 * format; imported, it starts afresh at its next push.
 * After an import, af_session_wire, af_session_levels and af_session_wire_first_frames are AF_ERR_INVALID until the next
 * push: the last push's outputs no longer describe the imported slots.
 * The caller frees a moved stream's old slot with af_session_reset_streams; growing a full session is importing all of
 * its streams into a larger one.  Device records cross GPUs by the caller's own copy (cudaMemcpyPeerAsync).
 * Both calls block until the records (export) or the slots (import) are complete.  With mem == AF_MEM_DEVICE the records
 * live on the session's GPU, and whatever produced them on other streams must have finished. */
/* Bytes of one stream record of this session (a multiple of 16).  Fixed for a session: it depends only on its framing. */
AF_API size_t af_session_stream_record_bytes(const af_session *s);
/* Snapshot: record i (records + i * record_bytes) receives the complete state of stream streams[i] (a stream may be listed
 * twice).  The session does not change.  mem: AF_MEM_HOST (any host memory) or AF_MEM_DEVICE (on the session's GPU).
 * AF_ERR_INVALID, before anything is written, for a stream index out of range, null arrays with n > 0 and a bad mem. */
AF_API int af_session_export_streams(af_session *s, const uint32_t *streams, size_t n, void *records, int mem);
/* Slot slots[i] continues the stream of record i; the slot's previous stream is discarded, as by
 * af_session_reset_streams.  format: NULL, or per record an index into B's formats with the record's rate and channel
 * count (NULL: the first admitted format with them).  AF_ERR_INVALID, before anything changes, for a bad magic or version,
 * a record size other than this session's, an incompatible framing or vad_enable, a rate and channel count no format
 * admits, a slot out of range or listed twice, an explicit format index out of range or whose rate or channels differ
 * from the record's, null arrays with n > 0 and a bad mem.  A session whose streams all stand at one position afterwards
 * runs its next equal-count push as the lockstep tick. */
AF_API int af_session_import_streams(af_session *s, const uint32_t *slots, const void *records, size_t n,
                                     const uint32_t *format, int mem);

#ifdef __cplusplus
}
#endif
#endif /* AUDIOFLOW_GPU_H */
