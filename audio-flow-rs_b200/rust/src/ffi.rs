//! Raw bindings to include/audioflow_gpu.h (what `bindgen` would emit, trimmed to the compat API).
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int};

#[repr(C)]
pub struct af_resampler { _p: [u8; 0] }
#[repr(C)]
pub struct af_batch_resampler { _p: [u8; 0] }
#[repr(C)]
pub struct af_vad { _p: [u8; 0] }

#[repr(C)]
#[derive(Clone, Copy)]
pub struct af_vad_config {
    pub threshold_db: f32,
    pub smoothing_factor: f32,
    pub silence_timeout_frames: u64,
    pub min_speech_frames: u64,
}

pub const AF_OK: c_int = 0;
pub const AF_FMT_F32: u16 = 0;
pub const AF_FMT_I16: u16 = 1;
pub const AF_MEM_DEVICE: c_int = 0;
pub const AF_MEM_HOST: c_int = 1;

// ---- the batched fast path (audioflow_gpu.h, "Batched fast path") ----
#[repr(C)] pub struct af_pipeline { _p: [u8; 0] }
#[repr(C)] pub struct af_batch { _p: [u8; 0] }
#[repr(C)] pub struct af_sharded_batch { _p: [u8; 0] }

#[repr(C)]
#[derive(Clone, Copy)]
pub struct af_pipeline_config {
    pub n_mels: u32,
    pub f_min: f32,
    pub f_max: f32,
    pub log_floor: f32,
    pub log10: u32,
    pub vad_enable: u32,
    pub vad: af_vad_config,
    pub vad_frame_len: u32,
    pub vad_hop: u32,
    pub write_pcm: u32,
    pub pcm16: u32,
}

#[repr(C)]
#[derive(Clone, Copy)]
pub struct af_stream_desc {
    pub data: *const std::os::raw::c_void,
    pub n_samples: u64,
    pub sample_rate: u32,
    pub channels: u16,
    pub format: u16,
}

#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct af_vad_final {
    pub smoothed_energy: f32,
    pub state: i32,
    pub silence_frames: u64,
    pub speech_frames: u64,
}

#[repr(C)]
pub struct af_outputs {
    pub pcm: *mut f32,
    pub pcm_stride: u64,
    pub logmel: *mut f32,
    pub logmel_stride: u64,
    pub vad: *mut u8,
    pub vad_stride: u64,
    pub energy: *mut f32,
    pub energy_stride: u64,
    pub vad_final: *mut af_vad_final,
}

#[repr(C)] pub struct af_ring { _private: [u8; 0] }
pub const AF_RING_EMPTY: c_int = -1;

// ---- streaming sessions (audioflow_gpu.h, "streaming sessions", level metering, wire output) ----
#[repr(C)] pub struct af_session { _p: [u8; 0] }

#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct af_wire_config {
    pub gate: u32,
    pub pcm16: u32,
    pub base64: u32,
    pub mem: i32,
}

#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct af_wire_tick {
    pub n_samples: u32,
    pub n_chars: u32,
    pub continued: u32,
    pub started: u16,
    pub ended: u16,
    pub in_speech: u8,
    pub pad: [u8; 3],
}

#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct af_stream_format {
    pub sample_rate: u32,
    pub channels: u16,
    pub pad: u16,
    pub max_tick_samples: u32,
}

extern "C" {
    pub fn af_session_create(p: *mut af_pipeline, n_streams: usize, sample_rate: u32, channels: u16, format: u16,
                             max_tick_samples: u32, out: *mut *mut af_session) -> c_int;
    pub fn af_session_destroy(s: *mut af_session);
    pub fn af_session_push(s: *mut af_session, data: *const std::os::raw::c_void, in_stride: u64, n_samples: u32, mem: c_int,
                           out: *const af_outputs, n_pcm: *mut u32, n_feat: *mut u32, n_vad: *mut u32) -> c_int;
    pub fn af_session_push_rings(s: *mut af_session, rings: *const *mut af_ring, n_samples: u32, out: *const af_outputs,
                                 n_pcm: *mut u32, n_feat: *mut u32, n_vad: *mut u32) -> c_int;
    pub fn af_session_reset(s: *mut af_session) -> c_int;
    pub fn af_session_enable_levels(s: *mut af_session, enable: c_int) -> c_int;
    pub fn af_session_levels(s: *const af_session, level_db: *mut f32, peak: *mut f32, is_speech: *mut u8) -> c_int;
    pub fn af_session_enable_wire(s: *mut af_session, cfg: *const af_wire_config) -> c_int;
    pub fn af_session_wire(s: *const af_session, pcm16: *mut *const i16, pcm16_stride: *mut u64, base64: *mut *const c_char,
                           base64_stride: *mut u64, ticks: *mut af_wire_tick, first_frame: *mut u64) -> c_int;
    pub fn af_session_push_streams(s: *mut af_session, data: *const std::os::raw::c_void, in_stride: u64, n_samples: *const u32,
                                   end: *const u8, mem: c_int, out: *const af_outputs,
                                   n_pcm: *mut u32, n_feat: *mut u32, n_vad: *mut u32) -> c_int;
    pub fn af_session_reset_streams(s: *mut af_session, streams: *const u32, n: usize) -> c_int;
    pub fn af_session_push_rings_available(s: *mut af_session, rings: *const *mut af_ring, max_samples: u32, end: *const u8,
                                           out: *const af_outputs, n_pcm: *mut u32, n_feat: *mut u32, n_vad: *mut u32) -> c_int;
    pub fn af_session_wire_first_frames(s: *const af_session, first_frame: *mut u64) -> c_int;
    pub fn af_session_create_formats(p: *mut af_pipeline, n_streams: usize, formats: *const af_stream_format, n_formats: usize,
                                     stream_format: *const u32, sample_format: u16, out: *mut *mut af_session) -> c_int;
    pub fn af_session_restart_streams(s: *mut af_session, streams: *const u32, format: *const u32, n: usize) -> c_int;
    pub fn af_session_set_vad_configs(s: *mut af_session, streams: *const u32, cfgs: *const af_vad_config, n: usize) -> c_int;
}

extern "C" {
    pub fn af_ring_create(capacity_samples: usize, out: *mut *mut af_ring) -> c_int;
    pub fn af_ring_destroy(r: *mut af_ring);
    pub fn af_ring_write(r: *mut af_ring, data: *const f32, n: usize) -> usize;
    pub fn af_ring_read(r: *mut af_ring, out: *mut f32, size: usize, n_read: *mut usize) -> c_int;
    pub fn af_ring_available(r: *const af_ring) -> usize;
    pub fn af_ring_clear(r: *mut af_ring);

    pub fn af_init(device: c_int) -> c_int;
    pub fn af_init_multi(n_gpus: c_int) -> c_int;
    pub fn af_device_count(count: *mut c_int) -> c_int;
    pub fn af_comm_size() -> c_int;
    pub fn af_shutdown() -> c_int;

    pub fn af_pipeline_config_default(cfg: *mut af_pipeline_config);
    pub fn af_pipeline_create(cfg: *const af_pipeline_config, out: *mut *mut af_pipeline) -> c_int;
    pub fn af_pipeline_destroy(p: *mut af_pipeline);
    pub fn af_batch_create(p: *mut af_pipeline, streams: *const af_stream_desc, n_streams: usize, mem: c_int,
                           out: *mut *mut af_batch) -> c_int;
    pub fn af_batch_destroy(b: *mut af_batch);
    pub fn af_batch_counts(b: *const af_batch, n_out: *mut u32, n_feat_frames: *mut u32, n_vad_frames: *mut u32) -> c_int;
    pub fn af_batch_strides(b: *const af_batch, pcm_stride: *mut u64, logmel_stride: *mut u64, vad_stride: *mut u64) -> c_int;
    pub fn af_batch_run_host(b: *mut af_batch, out: *const af_outputs) -> c_int;
    pub fn af_batch_set_vad_configs(b: *mut af_batch, cfgs: *const af_vad_config) -> c_int;

    pub fn af_sharded_batch_create(p: *mut af_pipeline, streams: *const af_stream_desc, n_streams: usize, mem: c_int,
                                   out: *mut *mut af_sharded_batch) -> c_int;
    pub fn af_sharded_batch_destroy(b: *mut af_sharded_batch);
    pub fn af_sharded_batch_shard(b: *const af_sharded_batch, rank: c_int, first: *mut usize, count: *mut usize,
                                  device: *mut c_int) -> c_int;
    pub fn af_sharded_batch_local(b: *mut af_sharded_batch, rank: c_int) -> *mut af_batch;
    pub fn af_sharded_batch_run_host(b: *mut af_sharded_batch, out: *const af_outputs) -> c_int;

    pub fn af_pcm16_encode(samples: *const f32, n: usize, out: *mut i16) -> c_int;
    pub fn af_pcm16_base64_len(n_samples: usize) -> usize;
    pub fn af_pcm16_base64(samples: *const f32, n: usize, out: *mut c_char, out_cap: usize, n_out: *mut usize) -> c_int;
    pub fn af_last_error(buf: *mut c_char, cap: usize) -> usize;

    pub fn af_to_mono(samples: *const f32, n_samples: usize, channels: u16, out: *mut f32, out_cap: usize,
                      n_out: *mut usize) -> c_int;

    pub fn af_resampler_create(input_rate: u32, output_rate: u32, out: *mut *mut af_resampler) -> c_int;
    pub fn af_resampler_destroy(r: *mut af_resampler);
    pub fn af_resampler_process(r: *mut af_resampler, input: *const f32, n: usize, out: *mut f32, out_cap: usize,
                                n_out: *mut usize) -> c_int;
    pub fn af_resample_max_output(input_rate: u32, output_rate: u32, n_in: usize) -> usize;

    pub fn af_batch_resampler_create(input_rate: u32, output_rate: u32, out: *mut *mut af_batch_resampler) -> c_int;
    pub fn af_batch_resampler_destroy(b: *mut af_batch_resampler);
    pub fn af_batch_resampler_process(b: *mut af_batch_resampler, input: *const f32, n: usize, out: *mut f32,
                                      out_cap: usize, n_out: *mut usize) -> c_int;
    pub fn af_batch_resampler_flush(b: *mut af_batch_resampler, out: *mut f32, out_cap: usize, n_out: *mut usize) -> c_int;

    pub fn af_vad_create(cfg: *const af_vad_config, out: *mut *mut af_vad) -> c_int;
    pub fn af_vad_destroy(v: *mut af_vad);
    pub fn af_vad_detect(v: *mut af_vad, frame: *const f32, n: usize, state: *mut u8) -> c_int;
    pub fn af_vad_reset(v: *mut af_vad) -> c_int;
    pub fn af_vad_state(v: *const af_vad) -> c_int;
    pub fn af_vad_energy_db(v: *const af_vad) -> f32;
    pub fn af_vad_is_speaking(v: *const af_vad) -> c_int;
    pub fn af_vad_speech_frame_count(v: *const af_vad) -> u64;
}
