//! The batched fast path behind the same crate: many independent `AudioFrame`s through
//! `to_mono -> BatchResampler(all) + flush -> STFT / log-mel -> framed VAD` in one call, on one GPU or sharded over
//! every GPU of the box (`MultiGpu`), and the wire payload of `WebSocketClient::send_audio`.  Results are identical to
//! driving the per-object types of `lib.rs` stream by stream (tests/test_parity_gpu.py::test_config1_reference_clip).
//!
//! Source only, like the rest of the crate: the graft build image has no Rust toolchain.
use crate::ffi;
use crate::{AudioError, AudioFrame, VadConfig, VadState};
use std::ptr;

fn check(rc: i32) -> Result<(), AudioError> {
    if rc == ffi::AF_OK { Ok(()) } else { Err(AudioError::ResamplingFailed(crate::last_error())) }
}

/// What one stream of a batch comes back as.
#[derive(Debug, Clone)]
pub struct StreamResult {
    /// resampled mono 16 kHz PCM (`BatchResampler::process` of the whole stream + `flush`)
    pub pcm: Vec<f32>,
    /// `[frame][mel]` log-mel rows (empty when `n_mels == 0`)
    pub logmel: Vec<f32>,
    pub n_mels: usize,
    /// `VoiceActivityDetector::detect` per 25 ms / 10 ms frame
    pub vad: Vec<VadState>,
    /// `speech_frame_count()` / `state()` after the last frame
    pub final_state: VadState,
    pub speech_frames: u64,
}

/// `af_pipeline`: feature geometry + VAD configuration shared by the batches built from it.
pub struct Pipeline { h: *mut ffi::af_pipeline, cfg: ffi::af_pipeline_config }
unsafe impl Send for Pipeline {}

impl Pipeline {
    /// `n_mels`: 0 (no features), 80 or 128; `vad`: `None` switches the detector off.
    pub fn new(n_mels: u32, vad: Option<VadConfig>) -> Result<Self, AudioError> {
        let mut cfg: ffi::af_pipeline_config = unsafe { std::mem::zeroed() };
        unsafe { ffi::af_pipeline_config_default(&mut cfg) };
        cfg.n_mels = n_mels;
        match vad {
            Some(v) => {
                cfg.vad_enable = 1;
                cfg.vad = vad_config_c(&v);
            }
            None => cfg.vad_enable = 0,
        }
        let mut h = ptr::null_mut();
        check(unsafe { ffi::af_pipeline_create(&cfg, &mut h) })?;
        Ok(Self { h, cfg })
    }

    /// One GPU (the calling thread's `af_init` device): host buffers in, host buffers out, blocking.
    pub fn process(&self, frames: &[AudioFrame]) -> Result<Vec<StreamResult>, AudioError> {
        let descs = descs_of(frames);
        let mut b = ptr::null_mut();
        check(unsafe { ffi::af_batch_create(self.h, descs.as_ptr(), descs.len(), ffi::AF_MEM_HOST, &mut b) })?;
        let r = self.run(frames.len(), |out| unsafe { ffi::af_batch_run_host(b, out) }, |no, nf, nv, ps, ls, vs| unsafe {
            let rc = ffi::af_batch_counts(b, no, nf, nv);
            if rc != ffi::AF_OK { return rc; }
            ffi::af_batch_strides(b, ps, ls, vs)
        });
        unsafe { ffi::af_batch_destroy(b) };
        r
    }

    /// `process` with one `VadConfig` per frame (each caller's `VoiceActivityDetector::new(config)`, vad.rs:80-88); the
    /// pipeline needs its detector on (`vad` not `None`).
    pub fn process_with_vad_configs(&self, frames: &[AudioFrame], vad: &[VadConfig]) -> Result<Vec<StreamResult>, AudioError> {
        if vad.len() != frames.len() {
            return Err(AudioError::ResamplingFailed(format!("{} frames and {} configurations", frames.len(), vad.len())));
        }
        let descs = descs_of(frames);
        let cfgs: Vec<ffi::af_vad_config> = vad.iter().map(vad_config_c).collect();
        let mut b = ptr::null_mut();
        check(unsafe { ffi::af_batch_create(self.h, descs.as_ptr(), descs.len(), ffi::AF_MEM_HOST, &mut b) })?;
        let r = check(unsafe { ffi::af_batch_set_vad_configs(b, cfgs.as_ptr()) }).and_then(|_| {
            self.run(frames.len(), |out| unsafe { ffi::af_batch_run_host(b, out) }, |no, nf, nv, ps, ls, vs| unsafe {
                let rc = ffi::af_batch_counts(b, no, nf, nv);
                if rc != ffi::AF_OK { return rc; }
                ffi::af_batch_strides(b, ps, ls, vs)
            })
        });
        unsafe { ffi::af_batch_destroy(b) };
        r
    }

    fn run(&self, n: usize, go: impl FnOnce(*const ffi::af_outputs) -> i32,
           geometry: impl FnOnce(*mut u32, *mut u32, *mut u32, *mut u64, *mut u64, *mut u64) -> i32)
           -> Result<Vec<StreamResult>, AudioError> {
        let (mut n_out, mut n_feat, mut n_vad) = (vec![0u32; n], vec![0u32; n], vec![0u32; n]);
        let (mut ps, mut ls, mut vs) = (0u64, 0u64, 0u64);
        check(geometry(n_out.as_mut_ptr(), n_feat.as_mut_ptr(), n_vad.as_mut_ptr(), &mut ps, &mut ls, &mut vs))?;
        let (ps, ls, vs) = (ps as usize, ls as usize, vs as usize);
        let mut pcm = vec![0.0f32; n * ps];
        let mut lm = vec![0.0f32; n * ls];
        let mut vad = vec![0u8; n * vs];
        let mut fin = vec![ffi::af_vad_final::default(); n];
        let out = ffi::af_outputs {
            pcm: pcm.as_mut_ptr(), pcm_stride: ps as u64,
            logmel: if self.cfg.n_mels != 0 { lm.as_mut_ptr() } else { ptr::null_mut() }, logmel_stride: ls as u64,
            vad: if self.cfg.vad_enable != 0 { vad.as_mut_ptr() } else { ptr::null_mut() }, vad_stride: vs as u64,
            energy: ptr::null_mut(), energy_stride: 0,
            vad_final: if self.cfg.vad_enable != 0 { fin.as_mut_ptr() } else { ptr::null_mut() },
        };
        check(go(&out))?;
        let m = self.cfg.n_mels as usize;
        Ok((0..n).map(|i| StreamResult {
            pcm: pcm[i * ps..i * ps + n_out[i] as usize].to_vec(),
            logmel: lm[i * ls..i * ls + n_feat[i] as usize * m].to_vec(),
            n_mels: m,
            vad: vad[i * vs..i * vs + if self.cfg.vad_enable != 0 { n_vad[i] as usize } else { 0 }]
                .iter().map(|&s| state_of(s as i32)).collect(),
            final_state: state_of(fin[i].state),
            speech_frames: fin[i].speech_frames,
        }).collect())
    }
}

impl Pipeline {
    /// the C handle, for the sessions of `stream.rs` built from this pipeline
    pub(crate) fn handle(&self) -> *mut ffi::af_pipeline { self.h }
    pub(crate) fn n_mels(&self) -> usize { self.cfg.n_mels as usize }
}

impl Drop for Pipeline {
    fn drop(&mut self) { unsafe { ffi::af_pipeline_destroy(self.h) } }
}

pub(crate) fn vad_config_c(v: &VadConfig) -> ffi::af_vad_config {
    ffi::af_vad_config {
        threshold_db: v.threshold_db,
        smoothing_factor: v.smoothing_factor,
        silence_timeout_frames: v.silence_timeout_frames as u64,
        min_speech_frames: v.min_speech_frames as u64,
    }
}

fn state_of(s: i32) -> VadState {
    match s { 1 => VadState::Speech, 2 => VadState::Ending, _ => VadState::Silence }
}

fn descs_of(frames: &[AudioFrame]) -> Vec<ffi::af_stream_desc> {
    frames.iter().map(|f| ffi::af_stream_desc {
        data: f.samples.as_ptr() as *const _,
        n_samples: f.samples.len() as u64,
        sample_rate: f.sample_rate,
        channels: f.channels,
        format: ffi::AF_FMT_F32,
    }).collect()
}

/// Every GPU of the box from ONE process: `af_init_multi` (one NCCL communicator inside the library), batches sharded by
/// input bytes, one host thread per GPU inside `af_sharded_batch_run_host`.
pub struct MultiGpu { n: i32 }

impl MultiGpu {
    /// `n_gpus == 0`: all of them.
    pub fn init(n_gpus: i32) -> Result<Self, AudioError> {
        let mut have = 0;
        check(unsafe { ffi::af_device_count(&mut have) })?;
        let n = if n_gpus <= 0 || n_gpus > have { have } else { n_gpus };
        check(unsafe { ffi::af_init_multi(n) })?;
        Ok(Self { n })
    }

    pub fn gpus(&self) -> i32 { self.n }

    pub fn process(&self, pipe: &Pipeline, frames: &[AudioFrame]) -> Result<Vec<StreamResult>, AudioError> {
        let descs = descs_of(frames);
        let mut sb = ptr::null_mut();
        check(unsafe { ffi::af_sharded_batch_create(pipe.h, descs.as_ptr(), descs.len(), ffi::AF_MEM_HOST, &mut sb) })?;
        let n_ranks = self.n;
        let r = pipe.run(frames.len(), |out| unsafe { ffi::af_sharded_batch_run_host(sb, out) }, |no, nf, nv, ps, ls, vs| unsafe {
            // per-rank batches hold the counts of their own streams; strides: the largest over the ranks
            for r in 0..n_ranks {
                let (mut first, mut count, mut dev) = (0usize, 0usize, -1);
                let rc = ffi::af_sharded_batch_shard(sb, r, &mut first, &mut count, &mut dev);
                if rc != ffi::AF_OK { return rc; }
                if count == 0 { continue; }
                let b = ffi::af_sharded_batch_local(sb, r);
                let rc = ffi::af_batch_counts(b, no.add(first), nf.add(first), nv.add(first));
                if rc != ffi::AF_OK { return rc; }
                let (mut a, mut l, mut v) = (0u64, 0u64, 0u64);
                let rc = ffi::af_batch_strides(b, &mut a, &mut l, &mut v);
                if rc != ffi::AF_OK { return rc; }
                *ps = (*ps).max(a); *ls = (*ls).max(l); *vs = (*vs).max(v);
            }
            ffi::AF_OK
        });
        unsafe { ffi::af_sharded_batch_destroy(sb) };
        r
    }
}

impl Drop for MultiGpu {
    fn drop(&mut self) { unsafe { ffi::af_shutdown(); } }
}

/// `(x.clamp(-1.0, 1.0) * 32767.0) as i16` per sample (websocket.rs:246-251).
pub fn pcm16_encode(samples: &[f32]) -> Result<Vec<i16>, AudioError> {
    let mut out = vec![0i16; samples.len()];
    check(unsafe { ffi::af_pcm16_encode(samples.as_ptr(), samples.len(), out.as_mut_ptr()) })?;
    Ok(out)
}

/// The `audio_base_64` field of `WebSocketClient::send_audio` / `MessageBuilder::audio_message`
/// (websocket.rs:244-254, :338-348): base64 of the little-endian PCM16 bytes.
pub fn pcm16_base64(samples: &[f32]) -> Result<String, AudioError> {
    let cap = unsafe { ffi::af_pcm16_base64_len(samples.len()) };
    let mut buf = vec![0u8; cap];
    let mut n = 0usize;
    check(unsafe { ffi::af_pcm16_base64(samples.as_ptr(), samples.len(), buf.as_mut_ptr() as *mut _, cap, &mut n) })?;
    buf.truncate(n);
    Ok(String::from_utf8(buf).expect("base64 is ASCII"))
}
