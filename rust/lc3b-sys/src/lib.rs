//! Raw bindings to `include/lc3b.h`.  Each function names the reference method it replaces.
#![no_std]
#![allow(non_camel_case_types)]
use core::ffi::{c_char, c_int, c_void};

pub const LC3B_OK: c_int = 0;
/// `Lc3DecoderError::Only16BitsPerAudioSampleSupported` (src/decoder/lc3_decoder.rs:80)
pub const LC3B_ERR_BITS_PER_SAMPLE: c_int = 1;
/// where the reference panics (bad channel index :228, slice-length asserts)
pub const LC3B_ERR_INVALID_ARG: c_int = 2;
pub const LC3B_ERR_CUDA: c_int = 3;
pub const LC3B_ERR_WORKSPACE: c_int = 4;

#[repr(C)]
pub struct lc3b_decoder {
    _private: [u8; 0],
}
#[repr(C)]
pub struct lc3b_encoder {
    _private: [u8; 0],
}
#[repr(C)]
pub struct lc3b_mixed_decoder {
    _private: [u8; 0],
}
#[repr(C)]
pub struct lc3b_sharded_decoder {
    _private: [u8; 0],
}
#[repr(C)]
pub struct lc3b_sharded_encoder {
    _private: [u8; 0],
}
/// one (sampling frequency, frame duration) bucket of a mixed-rate batch (`lc3b_mixed_bucket`)
#[repr(C)]
#[derive(Default, Clone, Copy, Debug)]
pub struct lc3b_mixed_bucket {
    pub sampling_frequency: i32,
    pub frame_duration: i32,
    pub first_row: i32,
    pub n_rows: i32,
    pub nf: i32,
    pub reserved: i32,
    pub host_pcm_offset: u64,
}
pub const LC3B_MIXED_MAX_BUCKETS: usize = 12;
/// int32 words of one inspection record (`lc3b_decoder_set_trace`); indices as the `LC3B_TR_*` enum of include/lc3b.h
pub const LC3B_TRACE_WORDS: usize = 48;
/// `Lc3Config` (src/common/config.rs:18-39)
#[repr(C)]
#[derive(Default, Clone, Copy, Debug)]
pub struct lc3b_config {
    pub fs_ind: i32,
    pub fs: i32,
    pub ne: i32,
    pub nb: i32,
    pub nf: i32,
    pub z: i32,
    pub n_ms: i32,
}

extern "C" {
    /// `Lc3Config::new` (src/common/config.rs:42)
    pub fn lc3b_config_new(sampling_frequency: c_int, frame_duration: c_int, out: *mut lc3b_config) -> c_int;
    pub fn lc3b_last_cuda_error() -> c_int;
    pub fn lc3b_version() -> *const c_char;

    /// `Lc3Decoder::calc_working_buffer_lengths` (src/decoder/lc3_decoder.rs:236)
    pub fn lc3b_decoder_workspace_bytes(n_streams: c_int, frame_duration: c_int, sampling_frequency: c_int,
                                        max_nbytes: c_int, device_bytes: *mut usize) -> c_int;
    /// `Lc3Decoder::new` (src/decoder/lc3_decoder.rs:181)
    pub fn lc3b_decoder_init(out: *mut *mut lc3b_decoder, n_streams: c_int, frame_duration: c_int,
                             sampling_frequency: c_int, max_nbytes: c_int, device: c_int, dev_workspace: *mut c_void,
                             workspace_bytes: usize, cuda_stream: *mut c_void) -> c_int;
    /// one `Lc3Decoder::decode_frame` (src/decoder/lc3_decoder.rs:217) per stream, device buffers
    pub fn lc3b_decode_frames(h: *mut lc3b_decoder, bits_per_sample: c_int, frames: *const u8, frame_nbytes: *const i32,
                              nbytes: c_int, frame_stride: usize, pcm_out: *mut i16, pcm_stride: usize,
                              status_out: *mut i32, cuda_stream: *mut c_void) -> c_int;
    /// same, host buffers (pinned => asynchronous)
    pub fn lc3b_decode_frames_host(h: *mut lc3b_decoder, bits_per_sample: c_int, frames: *const u8,
                                   frame_nbytes: *const i32, nbytes: c_int, frame_stride: usize, pcm_out: *mut i16,
                                   pcm_stride: usize, status_out: *mut i32, cuda_stream: *mut c_void) -> c_int;
    /// one `decode_frame` for each listed stream (`stream_ids`: host, `n_rows` distinct ids), device buffers by call row
    pub fn lc3b_decode_frames_subset(h: *mut lc3b_decoder, bits_per_sample: c_int, stream_ids: *const i32, n_rows: c_int,
                                     frames: *const u8, frame_nbytes: *const i32, nbytes: c_int, frame_stride: usize,
                                     pcm_out: *mut i16, pcm_stride: usize, status_out: *mut i32,
                                     cuda_stream: *mut c_void) -> c_int;
    /// the listed streams get the state `lc3b_decoder_init` gives a stream
    pub fn lc3b_decoder_reset_streams(h: *mut lc3b_decoder, stream_ids: *const i32, n: c_int, cuda_stream: *mut c_void) -> c_int;
    pub fn lc3b_decoder_set_host_pipelining(h: *mut lc3b_decoder, on: c_int) -> c_int;
    pub fn lc3b_decoder_host_fence(h: *mut lc3b_decoder, cuda_stream: *mut c_void) -> c_int;
    /// the frame loop of examples/decode.rs:85-123 as one call: `n_frames` frames of every stream (time-parallel)
    pub fn lc3b_decoder_multi_scratch_bytes(h: *const lc3b_decoder, n_frames: c_int, device_bytes: *mut usize) -> c_int;
    pub fn lc3b_decode_stream_frames(h: *mut lc3b_decoder, bits_per_sample: c_int, frames: *const u8, frame_nbytes: *const i32,
                                     nbytes: c_int, frame_stride: usize, n_frames: c_int, pcm_out: *mut i16,
                                     status_out: *mut i32, scratch: *mut c_void, scratch_bytes: usize,
                                     cuda_stream: *mut c_void) -> c_int;
    /// ragged time-parallel decode: `frame_counts[i]` frames of stream `stream_ids[i]` (host arrays of `n_rows`), units
    /// packed row after row in the caller's order
    pub fn lc3b_decoder_multi_subset_scratch_bytes(h: *const lc3b_decoder, n_rows: c_int, total_frames: i64,
                                                   device_bytes: *mut usize) -> c_int;
    pub fn lc3b_decode_stream_frames_subset(h: *mut lc3b_decoder, bits_per_sample: c_int, stream_ids: *const i32,
                                            frame_counts: *const i32, n_rows: c_int, frames: *const u8,
                                            frame_nbytes: *const i32, nbytes: c_int, frame_stride: usize, pcm_out: *mut i16,
                                            status_out: *mut i32, scratch: *mut c_void, scratch_bytes: usize,
                                            cuda_stream: *mut c_void) -> c_int;
    /// 0 = one launch per kernel, 1 = one cached CUDA graph per call
    pub fn lc3b_decoder_set_graph_mode(h: *mut lc3b_decoder, mode: c_int) -> c_int;
    pub fn lc3b_decoder_set_split(h: *mut lc3b_decoder, k: c_int) -> c_int;
    /// 0 = by batch size, 1 = warp-per-frame dequantisation kernel, 2 = thread-per-frame
    pub fn lc3b_decoder_set_dequant_mode(h: *mut lc3b_decoder, mode: c_int) -> c_int;
    /// promise: every frame is at least `min_nbytes` long or lost; lets the decoder drop dead LTPF history (include/lc3b.h)
    pub fn lc3b_decoder_set_min_nbytes(h: *mut lc3b_decoder, min_nbytes: c_int) -> c_int;
    pub fn lc3b_decoder_graph_stats(h: *const lc3b_decoder, hits: *mut u64, updates: *mut u64, builds: *mut u64) -> c_int;
    /// inspection: per-stream record of `LC3B_TRACE_WORDS` i32 and the entropy-decoded integer spectrum (device pointers)
    pub fn lc3b_decoder_set_trace(h: *mut lc3b_decoder, trace: *mut i32, x: *mut i32) -> c_int;
    pub fn lc3b_decoder_get_spectrum(h: *mut lc3b_decoder, out: *mut f32, cuda_stream: *mut c_void) -> c_int;
    pub fn lc3b_decoder_destroy(h: *mut lc3b_decoder);

    /// the set of reference decoders a mixed-rate population needs (`Lc3Decoder::new` takes ONE duration and ONE
    /// frequency, src/decoder/lc3_decoder.rs:181), driven as one batch; rows in bucket order
    pub fn lc3b_mixed_decoder_layout(n_streams: c_int, sampling_frequency: *const i32, frame_duration: *const i32,
                                     order: *mut i32, buckets: *mut lc3b_mixed_bucket, n_buckets: *mut i32,
                                     host_pcm_elems: *mut u64) -> c_int;
    pub fn lc3b_mixed_decoder_workspace_bytes(n_streams: c_int, sampling_frequency: *const i32, frame_duration: *const i32,
                                              max_nbytes: c_int, device_bytes: *mut usize) -> c_int;
    pub fn lc3b_mixed_decoder_init(out: *mut *mut lc3b_mixed_decoder, n_streams: c_int, sampling_frequency: *const i32,
                                   frame_duration: *const i32, max_nbytes: c_int, device: c_int, dev_workspace: *mut c_void,
                                   workspace_bytes: usize, cuda_stream: *mut c_void) -> c_int;
    pub fn lc3b_mixed_decode_frames(h: *mut lc3b_mixed_decoder, bits_per_sample: c_int, frames: *const u8,
                                    frame_nbytes: *const i32, nbytes: c_int, frame_stride: usize, pcm_out: *mut i16,
                                    pcm_stride: usize, status_out: *mut i32, cuda_stream: *mut c_void) -> c_int;
    pub fn lc3b_mixed_decode_frames_host(h: *mut lc3b_mixed_decoder, bits_per_sample: c_int, frames: *const u8,
                                         frame_nbytes: *const i32, nbytes: c_int, frame_stride: usize, pcm_out: *mut i16,
                                         status_out: *mut i32, cuda_stream: *mut c_void) -> c_int;
    pub fn lc3b_mixed_decoder_set_host_pipelining(h: *mut lc3b_mixed_decoder, on: c_int) -> c_int;
    pub fn lc3b_mixed_decoder_host_fence(h: *mut lc3b_mixed_decoder, cuda_stream: *mut c_void) -> c_int;
    pub fn lc3b_mixed_decoder_set_graph_mode(h: *mut lc3b_mixed_decoder, mode: c_int) -> c_int;
    pub fn lc3b_mixed_decoder_set_dequant_mode(h: *mut lc3b_mixed_decoder, mode: c_int) -> c_int;
    pub fn lc3b_mixed_decoder_destroy(h: *mut lc3b_mixed_decoder);

    /// one batch over the GPUs of a box: stream s -> shard floor(s * G / N); host buffers, one thread per GPU
    pub fn lc3b_sharded_decoder_create(out: *mut *mut lc3b_sharded_decoder, n_streams: c_int, frame_duration: c_int,
                                       sampling_frequency: c_int, max_nbytes: c_int, devices: *const c_int,
                                       n_devices: c_int) -> c_int;
    pub fn lc3b_sharded_decoder_n_shards(h: *const lc3b_sharded_decoder) -> c_int;
    pub fn lc3b_sharded_decoder_shard(h: *const lc3b_sharded_decoder, shard: c_int, device: *mut c_int,
                                      first_stream: *mut c_int, n_streams: *mut c_int) -> c_int;
    pub fn lc3b_sharded_decode_frames_host(h: *mut lc3b_sharded_decoder, bits_per_sample: c_int, frames: *const u8,
                                           frame_nbytes: *const i32, nbytes: c_int, frame_stride: usize, pcm_out: *mut i16,
                                           pcm_stride: usize, status_out: *mut i32) -> c_int;
    pub fn lc3b_sharded_decoder_wait(h: *mut lc3b_sharded_decoder) -> c_int;
    pub fn lc3b_sharded_decoder_set_min_nbytes(h: *mut lc3b_sharded_decoder, min_nbytes: c_int) -> c_int;
    pub fn lc3b_sharded_decoder_destroy(h: *mut lc3b_sharded_decoder);
    pub fn lc3b_sharded_encoder_create(out: *mut *mut lc3b_sharded_encoder, n_streams: c_int, frame_duration: c_int,
                                       sampling_frequency: c_int, max_nbytes: c_int, devices: *const c_int,
                                       n_devices: c_int) -> c_int;
    pub fn lc3b_sharded_encoder_n_shards(h: *const lc3b_sharded_encoder) -> c_int;
    pub fn lc3b_sharded_encoder_shard(h: *const lc3b_sharded_encoder, shard: c_int, device: *mut c_int,
                                      first_stream: *mut c_int, n_streams: *mut c_int) -> c_int;
    pub fn lc3b_sharded_encode_frames_host(h: *mut lc3b_sharded_encoder, pcm_in: *const i16, pcm_stride: usize,
                                           frames_out: *mut u8, nbytes: c_int, frame_stride: usize) -> c_int;
    pub fn lc3b_sharded_encoder_wait(h: *mut lc3b_sharded_encoder) -> c_int;
    pub fn lc3b_sharded_encoder_destroy(h: *mut lc3b_sharded_encoder);

    /// pinned, portable host memory for the host-buffer entry points
    pub fn lc3b_host_alloc(out: *mut *mut c_void, bytes: usize) -> c_int;
    pub fn lc3b_host_free(p: *mut c_void);

    /// `Lc3Encoder::calc_working_buffer_lengths` (src/encoder/lc3_encoder.rs:194)
    pub fn lc3b_encoder_workspace_bytes(n_streams: c_int, frame_duration: c_int, sampling_frequency: c_int,
                                        max_nbytes: c_int, device_bytes: *mut usize) -> c_int;
    /// `Lc3Encoder::new` (src/encoder/lc3_encoder.rs:117)
    pub fn lc3b_encoder_init(out: *mut *mut lc3b_encoder, n_streams: c_int, frame_duration: c_int,
                             sampling_frequency: c_int, max_nbytes: c_int, device: c_int, dev_workspace: *mut c_void,
                             workspace_bytes: usize, cuda_stream: *mut c_void) -> c_int;
    /// one `Lc3Encoder::encode_frame` (src/encoder/lc3_encoder.rs:175) per stream, device buffers
    pub fn lc3b_encode_frames(h: *mut lc3b_encoder, pcm_in: *const i16, pcm_stride: usize, frames_out: *mut u8,
                              nbytes: c_int, frame_stride: usize, cuda_stream: *mut c_void) -> c_int;
    /// same, host buffers
    pub fn lc3b_encode_frames_host(h: *mut lc3b_encoder, pcm_in: *const i16, pcm_stride: usize, frames_out: *mut u8,
                                   nbytes: c_int, frame_stride: usize, cuda_stream: *mut c_void) -> c_int;
    /// one `encode_frame` for each listed stream (`stream_ids`: host, `n_rows` distinct ids), device buffers by call row
    pub fn lc3b_encode_frames_subset(h: *mut lc3b_encoder, stream_ids: *const i32, n_rows: c_int, pcm_in: *const i16,
                                     pcm_stride: usize, frames_out: *mut u8, nbytes: c_int, frame_stride: usize,
                                     cuda_stream: *mut c_void) -> c_int;
    /// the listed streams get the state `lc3b_encoder_init` gives a stream
    pub fn lc3b_encoder_reset_streams(h: *mut lc3b_encoder, stream_ids: *const i32, n: c_int, cuda_stream: *mut c_void) -> c_int;
    pub fn lc3b_encoder_set_host_pipelining(h: *mut lc3b_encoder, on: c_int) -> c_int;
    /// the frame loop of examples/encode.rs:73-116 as one call: `n_frames` frames of every stream (time-parallel)
    pub fn lc3b_encoder_multi_scratch_bytes(h: *const lc3b_encoder, n_frames: c_int, device_bytes: *mut usize) -> c_int;
    pub fn lc3b_encode_stream_frames(h: *mut lc3b_encoder, pcm_in: *const i16, n_frames: c_int, frames_out: *mut u8,
                                     nbytes: c_int, frame_stride: usize, scratch: *mut c_void, scratch_bytes: usize,
                                     cuda_stream: *mut c_void) -> c_int;
    /// ragged time-parallel encode: `frame_counts[i]` frames of stream `stream_ids[i]` (host arrays of `n_rows`)
    pub fn lc3b_encoder_multi_subset_scratch_bytes(h: *const lc3b_encoder, n_rows: c_int, total_frames: i64,
                                                   device_bytes: *mut usize) -> c_int;
    pub fn lc3b_encode_stream_frames_subset(h: *mut lc3b_encoder, stream_ids: *const i32, frame_counts: *const i32,
                                            n_rows: c_int, pcm_in: *const i16, frames_out: *mut u8, nbytes: c_int,
                                            frame_stride: usize, scratch: *mut c_void, scratch_bytes: usize,
                                            cuda_stream: *mut c_void) -> c_int;
    pub fn lc3b_encoder_set_graph_mode(h: *mut lc3b_encoder, mode: c_int) -> c_int;
    pub fn lc3b_encoder_destroy(h: *mut lc3b_encoder);
}
