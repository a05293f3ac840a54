// audioflow.hpp -- C++17 host-side mirror of the reference's audio module
// (src-tauri/src/modules/audio/mod.rs:9-11) over the C ABI of libaudioflow_gpu.so.
// The reference is compiled code (Rust) whose toolchain is absent from the build image, so this
// header is the compiled-language stand-in for the Rust shim in ../rust: same type names, method
// names, argument meaning and error behaviour.  Header only; contains no arithmetic of the path.
#pragma once
#include <cmath>
#include <cstdint>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/audioflow_gpu.h"

namespace audioflow {

// AudioError::ResamplingFailed (src-tauri/src/error.rs:109-110)
struct ResamplingFailed : std::runtime_error {
    explicit ResamplingFailed(const std::string &m) : std::runtime_error("Resampling failed: " + m) {}
};

inline void check(int rc)
{
    if (rc == AF_OK) return;
    char buf[512];
    af_last_error(buf, sizeof(buf));
    throw ResamplingFailed(buf);
}

// capture.rs:11-42
struct AudioFrame {
    std::vector<float> samples;
    uint32_t sample_rate = 0;
    uint16_t channels = 1;
    unsigned __int128 timestamp_ns = 0;

    AudioFrame(std::vector<float> s, uint32_t rate, uint16_t ch, unsigned __int128 ts = 0)
        : samples(std::move(s)), sample_rate(rate), channels(ch), timestamp_ns(ts) {}

    AudioFrame to_mono() const
    {
        if (channels == 1) return *this;
        const size_t frames = (samples.size() + channels - 1) / channels;
        std::vector<float> mono(frames);
        size_t n = 0;
        check(af_to_mono(samples.data(), samples.size(), channels, mono.data(), frames, &n));
        mono.resize(n);
        return AudioFrame(std::move(mono), sample_rate, 1, timestamp_ns);
    }
};

// resampler.rs:12-112
class AudioResampler {
public:
    AudioResampler(uint32_t input_rate, uint32_t output_rate) : in_(input_rate), out_(output_rate)
    {
        check(af_resampler_create(input_rate, output_rate, &h_));
    }
    static AudioResampler create_48k_to_16k() { return AudioResampler(48000, 16000); }
    AudioResampler(AudioResampler &&o) noexcept : h_(o.h_), in_(o.in_), out_(o.out_) { o.h_ = nullptr; }
    AudioResampler(const AudioResampler &) = delete;
    ~AudioResampler() { if (h_) af_resampler_destroy(h_); }

    std::vector<float> process(const std::vector<float> &input)
    {
        std::vector<float> out(std::max(input.size(), af_resample_max_output(in_, out_, 128)));
        size_t n = 0;
        check(af_resampler_process(h_, input.data(), input.size(), out.data(), out.size(), &n));
        out.resize(n);
        return out;
    }
    uint32_t input_rate() const { return in_; }
    uint32_t output_rate() const { return out_; }
    bool needs_resampling() const { return in_ != out_; }

private:
    af_resampler *h_ = nullptr;
    uint32_t in_, out_;
};

// resampler.rs:115-166
class BatchResampler {
public:
    BatchResampler(uint32_t input_rate, uint32_t output_rate) : in_(input_rate), out_(output_rate)
    {
        check(af_batch_resampler_create(input_rate, output_rate, &h_));
    }
    BatchResampler(const BatchResampler &) = delete;
    ~BatchResampler() { if (h_) af_batch_resampler_destroy(h_); }
    std::vector<float> process(const std::vector<float> &input)
    {
        std::vector<float> out(af_resample_max_output(in_, out_, input.size() + 128));
        size_t n = 0;
        check(af_batch_resampler_process(h_, input.data(), input.size(), out.data(), out.size(), &n));
        out.resize(n);
        return out;
    }
    std::vector<float> flush()
    {
        std::vector<float> out(af_resample_max_output(in_, out_, 128));
        size_t n = 0;
        check(af_batch_resampler_flush(h_, out.data(), out.size(), &n));
        out.resize(n);
        return out;
    }

private:
    af_batch_resampler *h_ = nullptr;
    uint32_t in_, out_;
};

// capture.rs:84-161 -- the capture hand-off.  write() keeps one slot free and returns the count written; read() returns
// nothing (the reference's None) on an empty ring, else min(size, available) samples.
class RingBuffer {
public:
    explicit RingBuffer(size_t capacity_samples) { check(af_ring_create(capacity_samples, &h_)); capacity = af_ring_capacity(h_); }
    RingBuffer(const RingBuffer &) = delete;
    ~RingBuffer() { if (h_) af_ring_destroy(h_); }
    size_t write(const std::vector<float> &data) { return af_ring_write(h_, data.data(), data.size()); }
    bool read(size_t size, std::vector<float> *out)
    {
        out->assign(size, 0.0f);
        size_t n = 0;
        const int rc = af_ring_read(h_, out->data(), size, &n);
        if (rc == AF_RING_EMPTY) { out->clear(); return false; }
        check(rc);
        out->resize(n);
        return true;
    }
    size_t available() const { return af_ring_available(h_); }
    void clear() { af_ring_clear(h_); }
    af_ring *handle() { return h_; }
    size_t capacity = 0;

private:
    af_ring *h_ = nullptr;
};

// af_session: n lockstep streams with their state on the GPU between ticks; outputs of a tick go to caller rows `out`
// (af_outputs, may be null), the wire payloads and levels stay in the session until the next push.
struct WirePayload {
    std::vector<int16_t> pcm16;       // empty unless the PCM16 encoding is on (and the rows are host rows)
    std::string base64;               // the "audio_base_64" field of send_audio (websocket.rs:244-254)
    uint32_t continued = 0;
    uint16_t started = 0, ended = 0;
    bool in_speech = false;
};
struct TickCounts { std::vector<uint32_t> n_pcm, n_feat, n_vad; };

class Session {
public:
    Session(af_pipeline *p, size_t n_streams, uint32_t sample_rate, uint16_t channels, uint16_t format, uint32_t max_tick_samples)
        : n_(n_streams)
    {
        check(af_session_create(p, n_streams, sample_rate, channels, format, max_tick_samples, &h_));
    }
    // a session of stream_format.size() streams that admits `formats`; stream k starts in formats[stream_format[k]]
    Session(af_pipeline *p, const std::vector<af_stream_format> &formats, const std::vector<uint32_t> &stream_format,
            uint16_t sample_format)
        : n_(stream_format.size())
    {
        check(af_session_create_formats(p, n_, formats.data(), formats.size(), stream_format.data(), sample_format, &h_));
    }
    Session(const Session &) = delete;
    ~Session() { if (h_) af_session_destroy(h_); }

    TickCounts push(const void *data, uint64_t in_stride, uint32_t n_samples, int mem, const af_outputs *out = nullptr)
    {
        TickCounts c{std::vector<uint32_t>(n_), std::vector<uint32_t>(n_), std::vector<uint32_t>(n_)};
        check(af_session_push(h_, data, in_stride, n_samples, mem, out, c.n_pcm.data(), c.n_feat.data(), c.n_vad.data()));
        return c;
    }
    TickCounts push_rings(std::vector<RingBuffer *> &rings, uint32_t n_samples, const af_outputs *out = nullptr)
    {
        std::vector<af_ring *> hs;
        for (RingBuffer *r : rings) hs.push_back(r->handle());
        TickCounts c{std::vector<uint32_t>(n_), std::vector<uint32_t>(n_), std::vector<uint32_t>(n_)};
        check(af_session_push_rings(h_, hs.data(), n_samples, out, c.n_pcm.data(), c.n_feat.data(), c.n_vad.data()));
        return c;
    }
    void reset() { check(af_session_reset(h_)); }

    // independent stream timelines: stream k pushes n_samples[k] samples from row k (rows in_stride apart); end[k] != 0
    // (end may be empty) ends stream k after them (BatchResampler::flush); its next push starts afresh
    TickCounts push_streams(const void *data, uint64_t in_stride, const std::vector<uint32_t> &n_samples,
                            const std::vector<uint8_t> &end, int mem, const af_outputs *out = nullptr)
    {
        if (n_samples.size() != n_ || (!end.empty() && end.size() != n_)) throw std::invalid_argument("push_streams: one count and end flag per stream");
        TickCounts c{std::vector<uint32_t>(n_), std::vector<uint32_t>(n_), std::vector<uint32_t>(n_)};
        check(af_session_push_streams(h_, data, in_stride, n_samples.data(), end.empty() ? nullptr : end.data(), mem, out,
                                      c.n_pcm.data(), c.n_feat.data(), c.n_vad.data()));
        return c;
    }
    // AudioCapturer::read_frame(max) for every stream: what each ring holds, up to max_samples, in whole frames
    TickCounts push_rings_available(std::vector<RingBuffer *> &rings, uint32_t max_samples, const std::vector<uint8_t> &end = {},
                                    const af_outputs *out = nullptr)
    {
        if (rings.size() != n_ || (!end.empty() && end.size() != n_)) throw std::invalid_argument("push_rings_available: one ring and end flag per stream");
        std::vector<af_ring *> hs;
        for (RingBuffer *r : rings) hs.push_back(r->handle());
        TickCounts c{std::vector<uint32_t>(n_), std::vector<uint32_t>(n_), std::vector<uint32_t>(n_)};
        check(af_session_push_rings_available(h_, hs.data(), max_samples, end.empty() ? nullptr : end.data(), out,
                                              c.n_pcm.data(), c.n_feat.data(), c.n_vad.data()));
        return c;
    }
    // the listed streams start afresh at their next push, without a flush
    void reset_streams(const std::vector<uint32_t> &streams) { check(af_session_reset_streams(h_, streams.data(), streams.size())); }
    // the same, each stream starting in the session's format format[i]
    void restart_streams(const std::vector<uint32_t> &streams, const std::vector<uint32_t> &format)
    {
        if (streams.size() != format.size()) throw std::invalid_argument("restart_streams: one format per stream");
        check(af_session_restart_streams(h_, streams.data(), format.data(), streams.size()));
    }
    // stream streams[i] decides its frames from the next push on under cfgs[i] (VoiceActivityDetector::new(config) per
    // caller); the detector keeps its state and the configuration stays with the slot
    void set_vad_configs(const std::vector<uint32_t> &streams, const std::vector<af_vad_config> &cfgs)
    {
        if (streams.size() != cfgs.size()) throw std::invalid_argument("set_vad_configs: one configuration per stream");
        check(af_session_set_vad_configs(h_, streams.data(), cfgs.data(), streams.size()));
    }

    void enable_levels(bool on = true) { check(af_session_enable_levels(h_, on ? 1 : 0)); }
    // AudioLevel{level, peak} / VolumeLevel{level, is_speech} of the last tick, per stream
    void levels(std::vector<float> *level_db, std::vector<float> *peak, std::vector<uint8_t> *is_speech) const
    {
        level_db->resize(n_); peak->resize(n_); is_speech->resize(n_);
        check(af_session_levels(h_, level_db->data(), peak->data(), is_speech->data()));
    }

    // gate: only the hops of the VAD's speech frames; mem AF_MEM_HOST (payloads copied out by wire()) or AF_MEM_DEVICE
    void enable_wire(bool gate, bool pcm16 = true, bool base64 = true, int mem = AF_MEM_HOST)
    {
        const af_wire_config cfg{gate ? 1u : 0u, pcm16 ? 1u : 0u, base64 ? 1u : 0u, mem};
        check(af_session_enable_wire(h_, &cfg));
        wire_host_ = mem == AF_MEM_HOST;
    }
    void disable_wire() { check(af_session_enable_wire(h_, nullptr)); }
    std::vector<WirePayload> wire(uint64_t *first_frame = nullptr) const
    {
        const int16_t *pcm = nullptr;
        const char *b64 = nullptr;
        uint64_t ps = 0, bs = 0;
        std::vector<af_wire_tick> t(n_);
        check(af_session_wire(h_, &pcm, &ps, &b64, &bs, t.data(), first_frame));
        std::vector<WirePayload> out(n_);
        for (size_t k = 0; k < n_; ++k) {
            WirePayload &w = out[k];
            if (wire_host_ && pcm) w.pcm16.assign(pcm + k * ps, pcm + k * ps + t[k].n_samples);
            if (wire_host_ && b64) w.base64.assign(b64 + k * bs, t[k].n_chars);
            w.continued = t[k].continued; w.started = t[k].started; w.ended = t[k].ended; w.in_speech = t[k].in_speech != 0;
        }
        return out;
    }
    // per stream: the first frame completed by the last push, in the stream's own frame sequence since its last start
    std::vector<uint64_t> wire_first_frames() const
    {
        std::vector<uint64_t> f(n_);
        check(af_session_wire_first_frames(h_, f.data()));
        return f;
    }
    af_session *handle() { return h_; }

private:
    af_session *h_ = nullptr;
    size_t n_ = 0;
    bool wire_host_ = true;
};

// vad.rs:8-54
enum class VadLevel { Aggressive, Balanced, Relaxed };
enum class VadState { Silence = 0, Speech = 1, Ending = 2 };

struct VadConfig {
    float threshold_db = -50.0f;
    float smoothing_factor = 0.3f;
    size_t silence_timeout_frames = 15;
    size_t min_speech_frames = 3;
};

// vad.rs:60-205
class VoiceActivityDetector {
public:
    explicit VoiceActivityDetector(const VadConfig &c = VadConfig())
    {
        af_vad_config cc{c.threshold_db, c.smoothing_factor, c.silence_timeout_frames, c.min_speech_frames};
        check(af_vad_create(&cc, &h_));
    }
    VoiceActivityDetector(const VoiceActivityDetector &) = delete;
    ~VoiceActivityDetector() { if (h_) af_vad_destroy(h_); }
    VadState detect(const std::vector<float> &frame)
    {
        uint8_t s = 0;
        check(af_vad_detect(h_, frame.data(), frame.size(), &s));
        return static_cast<VadState>(s);
    }
    void reset() { check(af_vad_reset(h_)); }
    VadState state() const { return static_cast<VadState>(af_vad_state(h_)); }
    float energy_db() const { return af_vad_energy_db(h_); }
    bool is_speaking() const { return af_vad_is_speaking(h_) != 0; }
    size_t speech_frame_count() const { return af_vad_speech_frame_count(h_); }
    float calculate_energy(const std::vector<float> &frame) const
    {
        float e = 0;
        check(af_vad_frame_energy(frame.data(), frame.size(), &e));
        return e;
    }

private:
    af_vad *h_ = nullptr;
};

}  // namespace audioflow
