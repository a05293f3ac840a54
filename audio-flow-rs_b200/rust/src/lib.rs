//! Drop-in replacement for `src-tauri/src/modules/audio/{capture::AudioFrame, resampler, vad}`:
//! the same type names and method signatures (mod.rs:9-11 of the reference), every computation
//! forwarded to the CUDA library through the C ABI.  To switch the reference over:
//!
//! ```ignore
//! // src-tauri/src/modules/audio/mod.rs
//! pub use audioflow_gpu::{AudioFrame, AudioResampler, BatchResampler, VadConfig, VadLevel, VadState,
//!                         VoiceActivityDetector};
//! ```
//!
//! Source only: the graft build image has no Rust toolchain (see INTEGRATION.md).
mod ffi;
pub mod batch;
pub mod stream;

use std::ptr;

/// `AudioError` of src-tauri/src/error.rs:96-111 (the variants this path can produce).
#[derive(Debug, PartialEq, Eq, thiserror::Error)]
pub enum AudioError {
    #[error("Resampling failed: {0}")]
    ResamplingFailed(String),
}

fn last_error() -> String {
    let mut buf = vec![0u8; 512];
    unsafe { ffi::af_last_error(buf.as_mut_ptr() as *mut _, buf.len()) };
    let end = buf.iter().position(|&b| b == 0).unwrap_or(buf.len());
    String::from_utf8_lossy(&buf[..end]).into_owned()
}

fn check(rc: i32) -> Result<(), AudioError> {
    if rc == ffi::AF_OK { Ok(()) } else { Err(AudioError::ResamplingFailed(last_error())) }
}

/// capture.rs:11-42
#[derive(Debug, Clone)]
pub struct AudioFrame {
    pub samples: Vec<f32>,
    pub sample_rate: u32,
    pub channels: u16,
    pub timestamp_ns: u128,
}

impl AudioFrame {
    pub fn new(samples: Vec<f32>, sample_rate: u32, channels: u16, timestamp_ns: u128) -> Self {
        Self { samples, sample_rate, channels, timestamp_ns }
    }

    /// capture.rs:30-42; infallible in the reference, so a GPU failure panics here.
    pub fn to_mono(&self) -> Self {
        if self.channels == 1 {
            return self.clone();
        }
        let ch = self.channels as usize;
        let frames = (self.samples.len() + ch - 1) / ch;
        let mut mono = vec![0.0f32; frames];
        let mut n = 0usize;
        let rc = unsafe {
            ffi::af_to_mono(self.samples.as_ptr(), self.samples.len(), self.channels, mono.as_mut_ptr(), frames, &mut n)
        };
        check(rc).expect("af_to_mono");
        mono.truncate(n);
        Self::new(mono, self.sample_rate, 1, self.timestamp_ns)
    }
}

/// resampler.rs:12-112
pub struct AudioResampler {
    h: *mut ffi::af_resampler,
    input_rate: u32,
    output_rate: u32,
}
unsafe impl Send for AudioResampler {}

impl AudioResampler {
    pub fn new(input_rate: u32, output_rate: u32) -> Result<Self, AudioError> {
        let mut h = ptr::null_mut();
        check(unsafe { ffi::af_resampler_create(input_rate, output_rate, &mut h) })?;
        Ok(Self { h, input_rate, output_rate })
    }
    pub fn create_48k_to_16k() -> Result<Self, AudioError> { Self::new(48000, 16000) }

    pub fn process(&mut self, input: &[f32]) -> Result<Vec<f32>, AudioError> {
        if self.h.is_null() {
            // the `Default` fallback (resampler.rs:169-178: `resampler: None`) passes its input through (resampler.rs:72-75)
            return Ok(input.to_vec());
        }
        let cap = input.len().max(unsafe { ffi::af_resample_max_output(self.input_rate, self.output_rate, 128) });
        let mut out = vec![0.0f32; cap];
        let mut n = 0usize;
        check(unsafe { ffi::af_resampler_process(self.h, input.as_ptr(), input.len(), out.as_mut_ptr(), cap, &mut n) })?;
        out.truncate(n);
        Ok(out)
    }
    pub fn input_rate(&self) -> u32 { self.input_rate }
    pub fn output_rate(&self) -> u32 { self.output_rate }
    pub fn needs_resampling(&self) -> bool { self.input_rate != self.output_rate }
}

impl Drop for AudioResampler {
    fn drop(&mut self) { if !self.h.is_null() { unsafe { ffi::af_resampler_destroy(self.h) } } }
}

/// resampler.rs:169-178: `new(48000, 16000)`, and when that fails an object WITHOUT a resampler (it then passes its
/// input through) -- never a panic.
impl Default for AudioResampler {
    fn default() -> Self {
        Self::new(48000, 16000).unwrap_or_else(|_| Self { h: ptr::null_mut(), input_rate: 48000, output_rate: 16000 })
    }
}

/// resampler.rs:115-166
pub struct BatchResampler {
    h: *mut ffi::af_batch_resampler,
    input_rate: u32,
    output_rate: u32,
}
unsafe impl Send for BatchResampler {}

impl BatchResampler {
    pub fn new(input_rate: u32, output_rate: u32) -> Result<Self, AudioError> {
        let mut h = ptr::null_mut();
        check(unsafe { ffi::af_batch_resampler_create(input_rate, output_rate, &mut h) })?;
        Ok(Self { h, input_rate, output_rate })
    }
    pub fn process(&mut self, input: &[f32]) -> Result<Vec<f32>, AudioError> {
        let cap = unsafe { ffi::af_resample_max_output(self.input_rate, self.output_rate, input.len() + 128) };
        let mut out = vec![0.0f32; cap];
        let mut n = 0usize;
        check(unsafe { ffi::af_batch_resampler_process(self.h, input.as_ptr(), input.len(), out.as_mut_ptr(), cap, &mut n) })?;
        out.truncate(n);
        Ok(out)
    }
    pub fn flush(&mut self) -> Result<Vec<f32>, AudioError> {
        let cap = unsafe { ffi::af_resample_max_output(self.input_rate, self.output_rate, 128) };
        let mut out = vec![0.0f32; cap];
        let mut n = 0usize;
        check(unsafe { ffi::af_batch_resampler_flush(self.h, out.as_mut_ptr(), cap, &mut n) })?;
        out.truncate(n);
        Ok(out)
    }
}
impl Drop for BatchResampler {
    fn drop(&mut self) { unsafe { ffi::af_batch_resampler_destroy(self.h) } }
}

/// capture.rs:84-161 -- same `&self` methods as the reference (it locks internally); shared across threads with `Arc`.
pub struct RingBuffer {
    h: *mut ffi::af_ring,
    pub capacity: usize,
}
unsafe impl Send for RingBuffer {}
unsafe impl Sync for RingBuffer {}

impl RingBuffer {
    pub fn new(capacity_samples: usize) -> Self {
        let mut h = ptr::null_mut();
        let rc = unsafe { ffi::af_ring_create(capacity_samples, &mut h) };
        assert!(rc == 0, "RingBuffer::new({capacity_samples})");
        Self { h, capacity: capacity_samples }
    }
    pub fn write(&self, data: &[f32]) -> usize { unsafe { ffi::af_ring_write(self.h, data.as_ptr(), data.len()) } }
    pub fn read(&self, size: usize) -> Option<Vec<f32>> {
        let mut out = vec![0.0f32; size];
        let mut n = 0usize;
        let rc = unsafe { ffi::af_ring_read(self.h, out.as_mut_ptr(), size, &mut n) };
        if rc == ffi::AF_RING_EMPTY { return None; }
        out.truncate(n);
        Some(out)
    }
    pub fn available(&self) -> usize { unsafe { ffi::af_ring_available(self.h) } }
    pub fn clear(&self) { unsafe { ffi::af_ring_clear(self.h) } }
}
impl Drop for RingBuffer {
    fn drop(&mut self) { unsafe { ffi::af_ring_destroy(self.h) } }
}

/// vad.rs:8-17
#[derive(Debug, Clone, Copy, PartialEq, Eq, Default)]
pub enum VadLevel { #[default] Aggressive, Balanced, Relaxed }

/// vad.rs:21-43
#[derive(Debug, Clone, Copy)]
pub struct VadConfig {
    pub threshold_db: f32,
    pub smoothing_factor: f32,
    pub silence_timeout_frames: usize,
    pub min_speech_frames: usize,
}
impl Default for VadConfig {
    fn default() -> Self {
        Self { threshold_db: -50.0, smoothing_factor: 0.3, silence_timeout_frames: 15, min_speech_frames: 3 }
    }
}

/// vad.rs:47-54
#[derive(Debug, Clone, Copy, PartialEq, Eq)]
pub enum VadState { Silence, Speech, Ending }

fn state_from(v: i32) -> VadState {
    match v { 1 => VadState::Speech, 2 => VadState::Ending, _ => VadState::Silence }
}

/// vad.rs:60-205
#[derive(Debug)]
pub struct VoiceActivityDetector { h: *mut ffi::af_vad }
unsafe impl Send for VoiceActivityDetector {}

impl VoiceActivityDetector {
    pub fn new(config: VadConfig) -> Self {
        let c = ffi::af_vad_config {
            threshold_db: config.threshold_db,
            smoothing_factor: config.smoothing_factor,
            silence_timeout_frames: config.silence_timeout_frames as u64,
            min_speech_frames: config.min_speech_frames as u64,
        };
        let mut h = ptr::null_mut();
        check(unsafe { ffi::af_vad_create(&c, &mut h) }).expect("af_vad_create");
        Self { h }
    }
    pub fn detect(&mut self, frame: &[f32]) -> VadState {
        let mut s = 0u8;
        check(unsafe { ffi::af_vad_detect(self.h, frame.as_ptr(), frame.len(), &mut s) }).expect("af_vad_detect");
        state_from(s as i32)
    }
    pub fn reset(&mut self) { check(unsafe { ffi::af_vad_reset(self.h) }).expect("af_vad_reset") }
    pub fn state(&self) -> VadState { state_from(unsafe { ffi::af_vad_state(self.h) }) }
    pub fn energy_db(&self) -> f32 { unsafe { ffi::af_vad_energy_db(self.h) } }
    pub fn is_speaking(&self) -> bool { unsafe { ffi::af_vad_is_speaking(self.h) != 0 } }
    pub fn speech_frame_count(&self) -> usize { unsafe { ffi::af_vad_speech_frame_count(self.h) as usize } }
}
impl Default for VoiceActivityDetector {
    fn default() -> Self { Self::new(VadConfig::default()) }
}
impl Drop for VoiceActivityDetector {
    fn drop(&mut self) { unsafe { ffi::af_vad_destroy(self.h) } }
}

#[cfg(test)]
mod tests {
    //! The reference's own unit tests (capture.rs:371-400, resampler.rs:181-204, vad.rs:207-298), unchanged.
    use super::*;

    #[test]
    fn test_audio_frame_to_mono_stereo() {
        let frame = AudioFrame::new(vec![0.5, 0.25, -0.5, -0.25], 16000, 2, 1000);
        let mono = frame.to_mono();
        assert_eq!(mono.channels, 1);
        assert_eq!(mono.samples.len(), 2);
        assert!((mono.samples[0] - 0.375).abs() < 0.001);
        assert!((mono.samples[1] - (-0.375)).abs() < 0.001);
    }

    #[test]
    fn test_no_resample_needed() {
        let mut resampler = AudioResampler::new(16000, 16000).unwrap();
        let input = vec![0.1, 0.2, 0.3, 0.4];
        assert_eq!(resampler.process(&input).unwrap(), input);
    }

    #[test]
    fn test_vad_state_transitions() {
        let config = VadConfig { threshold_db: -50.0, silence_timeout_frames: 2, min_speech_frames: 1, smoothing_factor: 0.0 };
        let mut vad = VoiceActivityDetector::new(config);
        assert_eq!(vad.state(), VadState::Silence);
        let speech_frame = vec![0.5; 480];
        assert_eq!(vad.detect(&speech_frame), VadState::Speech);
        let silence_frame = vec![0.0001; 480];
        assert_eq!(vad.detect(&silence_frame), VadState::Speech);
        assert_eq!(vad.detect(&silence_frame), VadState::Ending);
        assert_eq!(vad.detect(&silence_frame), VadState::Silence);
    }
}
