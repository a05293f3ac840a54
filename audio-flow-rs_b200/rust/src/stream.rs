//! The streaming path of the desktop app: capture rings -> resample -> VAD -> drop the silence -> PCM16 -> base64, for
//! many streams per tick (`af_session_*`).  What the processing task calls before `WebSocketClient::send_audio`
//! (websocket.rs:244-254):
//!
//! ```ignore
//! let mut s = Session::new(&pipeline, rings.len(), 48000, 960, Some(WireGate::Speech))?;
//! loop {
//!     s.push_rings(&rings, 960)?;
//!     for (k, p) in s.wire()?.into_iter().enumerate() {
//!         if !p.audio_base_64.is_empty() { clients[k].send_audio(p.audio_base_64).await?; }
//!     }
//! }
//! ```
//!
//! Source only, like the rest of the crate (INTEGRATION.md).
use crate::batch::Pipeline;
use crate::ffi;
use crate::{AudioError, RingBuffer};
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

/// Counts of one tick, the same for every stream.
#[derive(Debug, Clone, Copy, Default)]
pub struct TickCounts { pub n_pcm: u32, pub n_feat: u32, pub n_vad: u32 }

/// `af_session`: n lockstep 16 kHz streams of one (rate, mono f32) with their state on the GPU between ticks.
pub struct Session { h: *mut ffi::af_session, n_streams: usize }
unsafe impl Send for Session {}

impl Session {
    /// `wire`: `None` for no wire output, else base64 payloads in pinned host rows, gated or not.
    pub fn new(pipeline: &Pipeline, n_streams: usize, sample_rate: u32, max_tick_samples: u32,
               wire: Option<WireGate>) -> Result<Self, AudioError> {
        let mut h = ptr::null_mut();
        check(unsafe { ffi::af_session_create(pipeline.handle(), n_streams, sample_rate, 1, ffi::AF_FMT_F32, max_tick_samples, &mut h) })?;
        let s = Self { h, n_streams };
        if let Some(g) = wire {
            let cfg = ffi::af_wire_config { gate: (g == WireGate::Speech) as u32, pcm16: 0, base64: 1, mem: ffi::AF_MEM_HOST };
            check(unsafe { ffi::af_session_enable_wire(s.h, &cfg) })?;
        }
        Ok(s)
    }

    /// `AudioCapturer::read_frame` (capture.rs:310-319) for every stream at once, pushed as one tick: takes exactly `n`
    /// samples from each ring (one ring per stream), nothing unless every ring holds them.
    pub fn push_rings(&mut self, rings: &[RingBuffer], n: u32) -> Result<TickCounts, AudioError> {
        if rings.len() != self.n_streams {
            return Err(AudioError::ResamplingFailed(format!("{} rings for {} streams", rings.len(), self.n_streams)));
        }
        let hs: Vec<*mut ffi::af_ring> = rings.iter().map(|r| r.h).collect();
        let mut c = TickCounts::default();
        check(unsafe { ffi::af_session_push_rings(self.h, hs.as_ptr(), n, ptr::null(), &mut c.n_pcm, &mut c.n_feat, &mut c.n_vad) })?;
        Ok(c)
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
