//! The streaming path of the desktop app: capture rings -> resample -> VAD -> drop the silence -> PCM16 -> base64, for
//! many streams per tick (`af_session_*`).  What the processing task calls before `WebSocketClient::send_audio`
//! (websocket.rs:244-254):
//!
//! ```ignore
//! let mut s = Session::new(&pipeline, rings.len(), 48000, 1920, Some(WireGate::Speech))?;
//! let mut ends = vec![false; rings.len()];
//! loop {
//!     // every stream takes what its capture callback delivered (up to 40 ms): a late callback stalls only its stream
//!     s.push_rings_available(&rings, 1920, &ends)?;
//!     for (k, p) in s.wire()?.into_iter().enumerate() {
//!         if !p.audio_base_64.is_empty() { clients[k].send_audio(p.audio_base_64).await?; }
//!     }
//!     // ends[k] = caller k hung up (the next tick flushes it, its slot then serves a new caller);
//!     // s.reset_streams(&[k]) drops a caller without a flush
//! }
//! ```
//!
//! Callers whose capture devices differ share one session through `Session::with_formats`; a freed slot takes a caller
//! with another device through `restart_streams`:
//!
//! ```ignore
//! let formats = [StreamFormat::new(48000, 1, 960), StreamFormat::new(44100, 2, 1764)];
//! let mut s = Session::with_formats(&pipeline, &formats, &device_format_of_each_caller, None)?;
//! // caller k hung up; a 44.1 kHz stereo caller takes its slot
//! s.restart_streams(&[k], &[1])?;
//! ```
//!
//! Source only, like the rest of the crate (INTEGRATION.md).
use crate::batch::Pipeline;
use crate::ffi;
use crate::{AudioError, RingBuffer, VadConfig};
use std::ptr;

fn check(rc: i32) -> Result<(), AudioError> {
    if rc == ffi::AF_OK { Ok(()) } else { Err(AudioError::ResamplingFailed(crate::last_error())) }
}

/// Which samples of a tick go on the wire.
#[derive(Debug, Clone, Copy, PartialEq, Eq)]
pub enum WireGate {
    /// every 16 kHz sample the tick produced
    All,
    /// only the hops of the frames of the VAD's speech segments (needs the VAD)
    Speech,
}

/// One stream's payload of one tick: the `audio_base_64` field of `send_audio` and the segment events of the tick.
#[derive(Debug, Clone, Default)]
pub struct WirePayload {
    pub audio_base_64: String,
    /// segments that started / were closed in this tick
    pub started: u16,
    pub ended: u16,
    /// the latest completed frame is Speech (`is_speaking()`)
    pub in_speech: bool,
    /// payload samples at the front that finish the segment open when the tick began (gated output only)
    pub continued: u32,
}

/// Counts of one stream in one tick (`push_rings` and `push_rings_available` return one per stream).
#[derive(Debug, Clone, Copy, Default)]
pub struct TickCounts { pub n_pcm: u32, pub n_feat: u32, pub n_vad: u32 }

/// One capture format of a session (`af_stream_format`): the device's rate and interleaved channel count, and the bound of
/// one tick's samples for a stream in it.
#[derive(Debug, Clone, Copy, PartialEq, Eq)]
pub struct StreamFormat { pub sample_rate: u32, pub channels: u16, pub max_tick_samples: u32 }

impl StreamFormat {
    pub fn new(sample_rate: u32, channels: u16, max_tick_samples: u32) -> Self { Self { sample_rate, channels, max_tick_samples } }
}

/// `af_session`: n 16 kHz streams (lockstep, or each on its own timeline) of f32 capture, each in one of the session's
/// formats (`new`: mono at one rate), with their state on the GPU between ticks.
pub struct Session { h: *mut ffi::af_session, n_streams: usize }
unsafe impl Send for Session {}

impl Session {
    /// `wire`: `None` for no wire output, else base64 payloads in pinned host rows, gated or not.
    pub fn new(pipeline: &Pipeline, n_streams: usize, sample_rate: u32, max_tick_samples: u32,
               wire: Option<WireGate>) -> Result<Self, AudioError> {
        let mut h = ptr::null_mut();
        check(unsafe { ffi::af_session_create(pipeline.handle(), n_streams, sample_rate, 1, ffi::AF_FMT_F32, max_tick_samples, &mut h) })?;
        Self { h, n_streams }.with_wire(wire)
    }

    /// A session of `stream_format.len()` streams that admits `formats`; stream k starts in `formats[stream_format[k]]`.
    pub fn with_formats(pipeline: &Pipeline, formats: &[StreamFormat], stream_format: &[u32],
                        wire: Option<WireGate>) -> Result<Self, AudioError> {
        let fs: Vec<ffi::af_stream_format> = formats.iter().map(|f| ffi::af_stream_format {
            sample_rate: f.sample_rate, channels: f.channels, pad: 0, max_tick_samples: f.max_tick_samples,
        }).collect();
        let mut h = ptr::null_mut();
        check(unsafe {
            ffi::af_session_create_formats(pipeline.handle(), stream_format.len(), fs.as_ptr(), fs.len(), stream_format.as_ptr(),
                                           ffi::AF_FMT_F32, &mut h)
        })?;
        Self { h, n_streams: stream_format.len() }.with_wire(wire)
    }

    fn with_wire(self, wire: Option<WireGate>) -> Result<Self, AudioError> {
        let s = self;
        if let Some(g) = wire {
            let cfg = ffi::af_wire_config { gate: (g == WireGate::Speech) as u32, pcm16: 0, base64: 1, mem: ffi::AF_MEM_HOST };
            check(unsafe { ffi::af_session_enable_wire(s.h, &cfg) })?;
        }
        Ok(s)
    }

    /// `AudioCapturer::read_frame` (capture.rs:310-319) for every stream at once, pushed as one tick: takes exactly `n`
    /// samples from each ring (one ring per stream), nothing unless every ring holds them.  Counts per stream (equal while
    /// the streams are in lockstep).
    pub fn push_rings(&mut self, rings: &[RingBuffer], n: u32) -> Result<Vec<TickCounts>, AudioError> {
        if rings.len() != self.n_streams {
            return Err(AudioError::ResamplingFailed(format!("{} rings for {} streams", rings.len(), self.n_streams)));
        }
        let hs: Vec<*mut ffi::af_ring> = rings.iter().map(|r| r.h).collect();
        let k = self.n_streams;
        let (mut p, mut f, mut v) = (vec![0u32; k], vec![0u32; k], vec![0u32; k]);
        check(unsafe {
            ffi::af_session_push_rings(self.h, hs.as_ptr(), n, ptr::null(), p.as_mut_ptr(), f.as_mut_ptr(), v.as_mut_ptr())
        })?;
        Ok((0..k).map(|i| TickCounts { n_pcm: p[i], n_feat: f[i], n_vad: v[i] }).collect())
    }

    /// `AudioCapturer::read_frame(max)` for every stream: each ring gives `min(max, available)` samples and the streams
    /// advance on their own timelines, so an empty ring stalls no other stream.  `ends[k]` (or an empty slice: none) ends
    /// stream k after its samples (`BatchResampler::flush`); its next push starts a new stream.  Counts per stream.
    pub fn push_rings_available(&mut self, rings: &[RingBuffer], max: u32, ends: &[bool]) -> Result<Vec<TickCounts>, AudioError> {
        if rings.len() != self.n_streams || (!ends.is_empty() && ends.len() != self.n_streams) {
            return Err(AudioError::ResamplingFailed(format!("{} rings and {} end flags for {} streams", rings.len(), ends.len(),
                                                            self.n_streams)));
        }
        let hs: Vec<*mut ffi::af_ring> = rings.iter().map(|r| r.h).collect();
        let e: Vec<u8> = ends.iter().map(|&b| b as u8).collect();
        let n = self.n_streams;
        let (mut p, mut f, mut v) = (vec![0u32; n], vec![0u32; n], vec![0u32; n]);
        check(unsafe {
            ffi::af_session_push_rings_available(self.h, hs.as_ptr(), max, if e.is_empty() { ptr::null() } else { e.as_ptr() },
                                                 ptr::null(), p.as_mut_ptr(), f.as_mut_ptr(), v.as_mut_ptr())
        })?;
        Ok((0..n).map(|k| TickCounts { n_pcm: p[k], n_feat: f[k], n_vad: v[k] }).collect())
    }

    /// The listed streams start afresh at their next push, without a flush (the caller went away); the others continue.
    pub fn reset_streams(&mut self, streams: &[u32]) -> Result<(), AudioError> {
        check(unsafe { ffi::af_session_reset_streams(self.h, streams.as_ptr(), streams.len()) })
    }

    /// `streams[i]` start afresh at their next push in the session's format `format[i]` (a new caller with another device).
    pub fn restart_streams(&mut self, streams: &[u32], format: &[u32]) -> Result<(), AudioError> {
        if streams.len() != format.len() {
            return Err(AudioError::ResamplingFailed(format!("{} streams and {} formats", streams.len(), format.len())));
        }
        check(unsafe { ffi::af_session_restart_streams(self.h, streams.as_ptr(), format.as_ptr(), streams.len()) })
    }

    /// Stream `streams[i]` decides every frame from the next push on under `cfgs[i]`: each caller's
    /// `VoiceActivityDetector::new(config)` (vad.rs:80-88).  The detector keeps its state; the configuration stays with
    /// the slot across resets, restarts and ends.
    pub fn set_vad_configs(&mut self, streams: &[u32], cfgs: &[VadConfig]) -> Result<(), AudioError> {
        if streams.len() != cfgs.len() {
            return Err(AudioError::ResamplingFailed(format!("{} streams and {} configurations", streams.len(), cfgs.len())));
        }
        let c: Vec<ffi::af_vad_config> = cfgs.iter().map(crate::batch::vad_config_c).collect();
        check(unsafe { ffi::af_session_set_vad_configs(self.h, streams.as_ptr(), c.as_ptr(), streams.len()) })
    }

    /// The payloads of the last tick, one per stream (valid until the next push; copied out here).
    pub fn wire(&self) -> Result<Vec<WirePayload>, AudioError> {
        let mut ticks = vec![ffi::af_wire_tick::default(); self.n_streams];
        let (mut b64, mut stride, mut first) = (ptr::null(), 0u64, 0u64);
        check(unsafe {
            ffi::af_session_wire(self.h, ptr::null_mut(), ptr::null_mut(), &mut b64, &mut stride, ticks.as_mut_ptr(), &mut first)
        })?;
        Ok(ticks.iter().enumerate().map(|(k, t)| {
            let text = unsafe { std::slice::from_raw_parts((b64 as *const u8).add(k * stride as usize), t.n_chars as usize) };
            WirePayload {
                audio_base_64: String::from_utf8_lossy(text).into_owned(),   // (base64 is ASCII)
                started: t.started,
                ended: t.ended,
                in_speech: t.in_speech != 0,
                continued: t.continued,
            }
        }).collect())
    }

    /// `AudioLevel` / `VolumeLevel` payloads of the last tick: (level_db, peak, is_speech) per stream.
    pub fn enable_levels(&mut self, on: bool) -> Result<(), AudioError> {
        check(unsafe { ffi::af_session_enable_levels(self.h, on as i32) })
    }
    pub fn levels(&self) -> Result<Vec<(f32, f32, bool)>, AudioError> {
        let n = self.n_streams;
        let (mut db, mut pk, mut sp) = (vec![0f32; n], vec![0f32; n], vec![0u8; n]);
        check(unsafe { ffi::af_session_levels(self.h, db.as_mut_ptr(), pk.as_mut_ptr(), sp.as_mut_ptr()) })?;
        Ok((0..n).map(|k| (db[k], pk[k], sp[k] != 0)).collect())
    }

    /// A fresh start for every stream (resampler position, frames, detector, open segments).
    pub fn reset(&mut self) -> Result<(), AudioError> { check(unsafe { ffi::af_session_reset(self.h) }) }
}

impl Drop for Session {
    fn drop(&mut self) { unsafe { ffi::af_session_destroy(self.h) } }
}
