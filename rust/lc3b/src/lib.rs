//! Batched drop-in for the hot path of ninjasource/lc3-codec:
//! `Lc3Decoder::decode_frame` (src/decoder/lc3_decoder.rs:217) and `Lc3Encoder::encode_frame`
//! (src/encoder/lc3_encoder.rs:175), one call per frame period for ALL streams.
//!
//! Preallocated-buffer style as in the reference: ask for the working-buffer size, allocate it yourself (device
//! memory, 256-byte aligned), lend it to `new` for `'a`.  Nothing is allocated on the device afterwards.
#![no_std]
use core::ffi::c_void;
use core::marker::PhantomData;
use core::ptr;
use lc3b_sys as sys;

/// `SamplingFrequency` (src/common/config.rs:2); discriminants are the C ABI's.
#[derive(Clone, Copy, Debug, PartialEq, Eq)]
#[repr(i32)]
pub enum SamplingFrequency {
    Hz8000 = 0,
    Hz16000 = 1,
    Hz24000 = 2,
    Hz32000 = 3,
    Hz44100 = 4,
    Hz48000 = 5,
}
/// `FrameDuration` (src/common/config.rs:12)
#[derive(Clone, Copy, Debug, PartialEq, Eq)]
#[repr(i32)]
pub enum FrameDuration {
    SevenPointFiveMs = 0,
    TenMs = 1,
}

/// `Lc3DecoderError` (src/decoder/lc3_decoder.rs:36-41); bitstream errors are concealed like the reference (:138-141).
#[derive(Debug, PartialEq, Eq)]
pub enum Lc3DecoderError {
    Only16BitsPerAudioSampleSupported,
}
/// `Lc3EncoderError` is empty in the reference (src/encoder/lc3_encoder.rs:30): encoding cannot fail.
#[derive(Debug)]
pub enum Lc3EncoderError {}

/// A caller-owned device allocation (any CUDA binding can produce the pointer).
pub struct DeviceBuf<'a> {
    pub ptr: *mut c_void,
    pub bytes: usize,
    pub _owner: PhantomData<&'a mut [u8]>,
}

/// Where a call's I/O buffers live.
#[derive(Clone, Copy)]
pub enum Residency {
    /// device pointers: asynchronous on the stream, no copies
    Device,
    /// host pointers (pinned => asynchronous): the library stages H2D / D2H itself
    Host,
}

fn check(rc: i32, what: &str) {
    // LC3B_ERR_INVALID_ARG stands where the reference panics; CUDA / workspace failures have no reference analogue
    if rc != sys::LC3B_OK {
        panic!("lc3b: {} failed with status {} (cuda error {})", what, rc, unsafe { sys::lc3b_last_cuda_error() });
    }
}

pub struct Lc3BatchDecoder<'a> {
    h: *mut sys::lc3b_decoder,
    n_streams: usize,
    nf: usize,
    stream: *mut c_void,
    _ws: PhantomData<&'a mut [u8]>,
}

impl<'a> Lc3BatchDecoder<'a> {
    /// `Lc3Decoder::calc_working_buffer_lengths` (:236): bytes of device working memory for `num_streams` channels.
    pub fn calc_working_buffer_lengths(num_streams: usize, duration: FrameDuration, freq: SamplingFrequency,
                                       max_nbytes: usize) -> usize {
        let mut n = 0usize;
        check(unsafe { sys::lc3b_decoder_workspace_bytes(num_streams as i32, duration as i32, freq as i32, max_nbytes as i32, &mut n) },
              "lc3b_decoder_workspace_bytes");
        n
    }

    /// `Lc3Decoder::new` (:181): borrows the working buffer for `'a`; state starts zeroed.
    pub fn new(num_streams: usize, duration: FrameDuration, freq: SamplingFrequency, working: DeviceBuf<'a>,
               max_nbytes: usize, device: i32, cuda_stream: *mut c_void) -> Self {
        let mut cfg = sys::lc3b_config::default();
        check(unsafe { sys::lc3b_config_new(freq as i32, duration as i32, &mut cfg) }, "lc3b_config_new");
        let mut h = ptr::null_mut();
        check(unsafe { sys::lc3b_decoder_init(&mut h, num_streams as i32, duration as i32, freq as i32, max_nbytes as i32,
                                              device, working.ptr, working.bytes, cuda_stream) }, "lc3b_decoder_init");
        Self { h, n_streams: num_streams, nf: cfg.nf as usize, stream: cuda_stream, _ws: PhantomData }
    }

    /// `decode_frame` for every stream: `frames[s*stride .. s*stride + nbytes]` -> `samples_out[s*nf .. (s+1)*nf]`.
    /// `frame_nbytes` (optional, same residency) gives per-stream lengths; 0 = lost frame (concealed).
    ///
    /// # Safety
    /// The pointers must be valid for the stated extents in the stated residency until the stream has drained.
    pub unsafe fn decode_frames(&mut self, num_bits_per_audio_sample: usize, residency: Residency, frames: *const u8,
                                frame_nbytes: *const i32, nbytes: usize, stride: usize, samples_out: *mut i16)
                                -> Result<(), Lc3DecoderError> {
        let f = match residency {
            Residency::Device => sys::lc3b_decode_frames,
            Residency::Host => sys::lc3b_decode_frames_host,
        };
        match f(self.h, num_bits_per_audio_sample as i32, frames, frame_nbytes, nbytes as i32, stride, samples_out, self.nf,
                ptr::null_mut(), self.stream) {
            sys::LC3B_OK => Ok(()),
            sys::LC3B_ERR_BITS_PER_SAMPLE => Err(Lc3DecoderError::Only16BitsPerAudioSampleSupported),
            rc => { check(rc, "lc3b_decode_frames"); unreachable!() }
        }
    }

    /// `decode_frames` that also reports which streams were concealed: `status_out[s]` = 0 decoded, 1 concealed.
    /// An extension - the reference swallows bitstream errors (src/decoder/lc3_decoder.rs:138-141).
    ///
    /// # Safety
    /// As for `decode_frames`; `status_out` has `num_streams` elements in the same residency.
    pub unsafe fn decode_frames_with_status(&mut self, num_bits_per_audio_sample: usize, residency: Residency,
                                            frames: *const u8, frame_nbytes: *const i32, nbytes: usize, stride: usize,
                                            samples_out: *mut i16, status_out: *mut i32) -> Result<(), Lc3DecoderError> {
        let f = match residency {
            Residency::Device => sys::lc3b_decode_frames,
            Residency::Host => sys::lc3b_decode_frames_host,
        };
        match f(self.h, num_bits_per_audio_sample as i32, frames, frame_nbytes, nbytes as i32, stride, samples_out, self.nf,
                status_out, self.stream) {
            sys::LC3B_OK => Ok(()),
            sys::LC3B_ERR_BITS_PER_SAMPLE => Err(Lc3DecoderError::Only16BitsPerAudioSampleSupported),
            rc => { check(rc, "lc3b_decode_frames"); unreachable!() }
        }
    }

    /// `decode_frame` (:217) for the listed streams only; every other stream is untouched.  Row i of the device buffers
    /// (`frames`, `samples_out`, `frame_nbytes`) belongs to stream `stream_ids[i]`: ids in `0..num_streams`, none twice
    /// (a bad list panics, like the reference's bad `channel_index`, :228).  `stream_ids` is only read during the call.
    ///
    /// # Safety
    /// As for `decode_frames`, with `stream_ids.len()` rows in device memory.
    pub unsafe fn decode_frames_subset(&mut self, num_bits_per_audio_sample: usize, stream_ids: &[i32], frames: *const u8,
                                       frame_nbytes: *const i32, nbytes: usize, stride: usize, samples_out: *mut i16)
                                       -> Result<(), Lc3DecoderError> {
        match sys::lc3b_decode_frames_subset(self.h, num_bits_per_audio_sample as i32, stream_ids.as_ptr(), stream_ids.len() as i32,
                                             frames, frame_nbytes, nbytes as i32, stride, samples_out, self.nf, ptr::null_mut(),
                                             self.stream) {
            sys::LC3B_OK => Ok(()),
            sys::LC3B_ERR_BITS_PER_SAMPLE => Err(Lc3DecoderError::Only16BitsPerAudioSampleSupported),
            rc => { check(rc, "lc3b_decode_frames_subset"); unreachable!() }
        }
    }

    /// The listed streams start over with the state `Lc3Decoder::new` gives a channel; no other stream is touched.
    pub fn reset_streams(&mut self, stream_ids: &[i32]) {
        check(unsafe { sys::lc3b_decoder_reset_streams(self.h, stream_ids.as_ptr(), stream_ids.len() as i32, self.stream) },
              "lc3b_decoder_reset_streams");
    }

    /// Bytes of caller-owned device scratch `decode_stream_frames` needs for `n_frames` frames per stream.
    pub fn multi_scratch_bytes(&self, n_frames: usize) -> usize {
        let mut n = 0usize;
        check(unsafe { sys::lc3b_decoder_multi_scratch_bytes(self.h, n_frames as i32, &mut n) }, "lc3b_decoder_multi_scratch_bytes");
        n
    }

    /// The frame loop of examples/decode.rs:85-123 as ONE call: `n_frames` consecutive frames of every stream
    /// (time-parallel).  Same PCM and same per-stream state afterwards as `n_frames` calls of `decode_frames`.
    /// Device buffers: `frames` is `[num_streams][n_frames][nbytes]`, `samples_out` is `[num_streams][n_frames * nf]`,
    /// `frame_nbytes` / `status_out` (nullable) are `[num_streams][n_frames]`.
    ///
    /// # Safety
    /// Device pointers valid for the stated extents until the stream has drained.
    pub unsafe fn decode_stream_frames(&mut self, num_bits_per_audio_sample: usize, frames: *const u8,
                                       frame_nbytes: *const i32, nbytes: usize, n_frames: usize, samples_out: *mut i16,
                                       status_out: *mut i32, scratch: DeviceBuf<'_>) -> Result<(), Lc3DecoderError> {
        match sys::lc3b_decode_stream_frames(self.h, num_bits_per_audio_sample as i32, frames, frame_nbytes, nbytes as i32,
                                             nbytes, n_frames as i32, samples_out, status_out, scratch.ptr, scratch.bytes,
                                             self.stream) {
            sys::LC3B_OK => Ok(()),
            sys::LC3B_ERR_BITS_PER_SAMPLE => Err(Lc3DecoderError::Only16BitsPerAudioSampleSupported),
            rc => { check(rc, "lc3b_decode_stream_frames"); unreachable!() }
        }
    }

    /// Bytes of caller-owned device scratch `decode_stream_frames_subset` needs for `n_rows` rows and `total_frames` frames.
    pub fn multi_subset_scratch_bytes(&self, n_rows: usize, total_frames: usize) -> usize {
        let mut n = 0usize;
        check(unsafe { sys::lc3b_decoder_multi_subset_scratch_bytes(self.h, n_rows as i32, total_frames as i64, &mut n) },
              "lc3b_decoder_multi_subset_scratch_bytes");
        n
    }

    /// `frame_counts[i]` consecutive frames of stream `stream_ids[i]` in ONE call (files of different lengths, jitter
    /// buffers of different depths); the same PCM and state as that many `decode_frames` calls on each listed stream,
    /// every other stream untouched.  Device buffers hold the frames packed row after row in the caller's order
    /// (`total` = sum of the counts): `frames` `[total][nbytes]`, `samples_out` `[total * nf]`, `frame_nbytes` /
    /// `status_out` (nullable) `[total]`.
    ///
    /// # Safety
    /// Device pointers valid for the stated extents until the stream has drained.
    pub unsafe fn decode_stream_frames_subset(&mut self, num_bits_per_audio_sample: usize, stream_ids: &[i32],
                                              frame_counts: &[i32], frames: *const u8, frame_nbytes: *const i32, nbytes: usize,
                                              samples_out: *mut i16, status_out: *mut i32, scratch: DeviceBuf<'_>)
                                              -> Result<(), Lc3DecoderError> {
        assert_eq!(stream_ids.len(), frame_counts.len(), "one frame count per stream id");
        match sys::lc3b_decode_stream_frames_subset(self.h, num_bits_per_audio_sample as i32, stream_ids.as_ptr(),
                                                    frame_counts.as_ptr(), stream_ids.len() as i32, frames, frame_nbytes,
                                                    nbytes as i32, nbytes, samples_out, status_out, scratch.ptr, scratch.bytes,
                                                    self.stream) {
            sys::LC3B_OK => Ok(()),
            sys::LC3B_ERR_BITS_PER_SAMPLE => Err(Lc3DecoderError::Only16BitsPerAudioSampleSupported),
            rc => { check(rc, "lc3b_decode_stream_frames_subset"); unreachable!() }
        }
    }

    /// Issue every call as one cached CUDA graph (`true`) or one launch per kernel (`false`); results are identical.
    pub fn set_graph_mode(&mut self, on: bool) {
        check(unsafe { sys::lc3b_decoder_set_graph_mode(self.h, on as i32) }, "lc3b_decoder_set_graph_mode");
    }

    /// Cut every call into `k` independent sub-batches whose kernels overlap (0 = by batch size, 1 = never, 2, 4).
    pub fn set_split(&mut self, k: i32) {
        check(unsafe { sys::lc3b_decoder_set_split(self.h, k) }, "lc3b_decoder_set_split");
    }

    /// Raw handle, for the inspection hooks of `lc3b_sys` (tests).
    pub fn raw(&mut self) -> *mut sys::lc3b_decoder { self.h }

    /// Let the PCM copy of call i overlap the kernels of call i+1 (host residency only); see `host_fence`.
    pub fn set_host_pipelining(&mut self, on: bool) {
        check(unsafe { sys::lc3b_decoder_set_host_pipelining(self.h, on as i32) }, "lc3b_decoder_set_host_pipelining");
    }
    /// Makes the stream wait for every outstanding pipelined PCM copy.
    pub fn host_fence(&mut self) {
        check(unsafe { sys::lc3b_decoder_host_fence(self.h, self.stream) }, "lc3b_decoder_host_fence");
    }
    pub fn num_streams(&self) -> usize { self.n_streams }
    pub fn samples_per_frame(&self) -> usize { self.nf }
}
impl Drop for Lc3BatchDecoder<'_> {
    fn drop(&mut self) { unsafe { sys::lc3b_decoder_destroy(self.h) } }
}

pub struct Lc3BatchEncoder<'a> {
    h: *mut sys::lc3b_encoder,
    n_streams: usize,
    nf: usize,
    stream: *mut c_void,
    _ws: PhantomData<&'a mut [u8]>,
}

impl<'a> Lc3BatchEncoder<'a> {
    /// `Lc3Encoder::calc_working_buffer_lengths` (src/encoder/lc3_encoder.rs:194).  Panics at 8 kHz like `Lc3Encoder::new`
    /// (bandwidth_detector.rs:42-56).
    pub fn calc_working_buffer_lengths(num_streams: usize, duration: FrameDuration, freq: SamplingFrequency,
                                       max_nbytes: usize) -> usize {
        let mut n = 0usize;
        check(unsafe { sys::lc3b_encoder_workspace_bytes(num_streams as i32, duration as i32, freq as i32, max_nbytes as i32, &mut n) },
              "lc3b_encoder_workspace_bytes");
        n
    }
    /// `Lc3Encoder::new` (:117)
    pub fn new(num_streams: usize, duration: FrameDuration, freq: SamplingFrequency, working: DeviceBuf<'a>,
               max_nbytes: usize, device: i32, cuda_stream: *mut c_void) -> Self {
        let mut cfg = sys::lc3b_config::default();
        check(unsafe { sys::lc3b_config_new(freq as i32, duration as i32, &mut cfg) }, "lc3b_config_new");
        let mut h = ptr::null_mut();
        check(unsafe { sys::lc3b_encoder_init(&mut h, num_streams as i32, duration as i32, freq as i32, max_nbytes as i32,
                                              device, working.ptr, working.bytes, cuda_stream) }, "lc3b_encoder_init");
        Self { h, n_streams: num_streams, nf: cfg.nf as usize, stream: cuda_stream, _ws: PhantomData }
    }
    /// `encode_frame` (:175) for every stream: `samples_in[s*nf ..]` -> `buf_out[s*stride .. s*stride + nbytes]`.
    ///
    /// # Safety
    /// As for `Lc3BatchDecoder::decode_frames`.
    pub unsafe fn encode_frames(&mut self, residency: Residency, samples_in: *const i16, buf_out: *mut u8, nbytes: usize,
                                stride: usize) -> Result<(), Lc3EncoderError> {
        let f = match residency {
            Residency::Device => sys::lc3b_encode_frames,
            Residency::Host => sys::lc3b_encode_frames_host,
        };
        check(f(self.h, samples_in, self.nf, buf_out, nbytes as i32, stride, self.stream), "lc3b_encode_frames");
        Ok(())
    }

    /// `encode_frame` (:175) for the listed streams only: row i of the device buffers belongs to stream `stream_ids[i]`
    /// (ids in `0..num_streams`, none twice; only read during the call).
    ///
    /// # Safety
    /// As for `encode_frames`, with `stream_ids.len()` rows in device memory.
    pub unsafe fn encode_frames_subset(&mut self, stream_ids: &[i32], samples_in: *const i16, buf_out: *mut u8, nbytes: usize,
                                       stride: usize) -> Result<(), Lc3EncoderError> {
        check(sys::lc3b_encode_frames_subset(self.h, stream_ids.as_ptr(), stream_ids.len() as i32, samples_in, self.nf, buf_out,
                                             nbytes as i32, stride, self.stream), "lc3b_encode_frames_subset");
        Ok(())
    }

    /// The listed streams start over with the state `Lc3Encoder::new` gives a channel; no other stream is touched.
    pub fn reset_streams(&mut self, stream_ids: &[i32]) {
        check(unsafe { sys::lc3b_encoder_reset_streams(self.h, stream_ids.as_ptr(), stream_ids.len() as i32, self.stream) },
              "lc3b_encoder_reset_streams");
    }

    /// Bytes of caller-owned device scratch `encode_stream_frames` needs for `n_frames` frames per stream.
    pub fn multi_scratch_bytes(&self, n_frames: usize) -> usize {
        let mut n = 0usize;
        check(unsafe { sys::lc3b_encoder_multi_scratch_bytes(self.h, n_frames as i32, &mut n) }, "lc3b_encoder_multi_scratch_bytes");
        n
    }

    /// The frame loop of examples/encode.rs:73-116 as ONE call: `n_frames` consecutive frames of every stream
    /// (time-parallel).  Same bytes and same per-stream state afterwards as `n_frames` calls of `encode_frames`.
    /// Device buffers: `samples_in` is `[num_streams][n_frames * nf]`; frame f of stream s goes to
    /// `buf_out[(s * n_frames + f) * stride ..][.. nbytes]`.
    ///
    /// # Safety
    /// Device pointers valid for the stated extents until the stream has drained.
    pub unsafe fn encode_stream_frames(&mut self, samples_in: *const i16, n_frames: usize, buf_out: *mut u8, nbytes: usize,
                                       stride: usize, scratch: DeviceBuf<'_>) -> Result<(), Lc3EncoderError> {
        check(sys::lc3b_encode_stream_frames(self.h, samples_in, n_frames as i32, buf_out, nbytes as i32, stride, scratch.ptr,
                                             scratch.bytes, self.stream), "lc3b_encode_stream_frames");
        Ok(())
    }

    /// Bytes of caller-owned device scratch `encode_stream_frames_subset` needs for `n_rows` rows and `total_frames` frames.
    pub fn multi_subset_scratch_bytes(&self, n_rows: usize, total_frames: usize) -> usize {
        let mut n = 0usize;
        check(unsafe { sys::lc3b_encoder_multi_subset_scratch_bytes(self.h, n_rows as i32, total_frames as i64, &mut n) },
              "lc3b_encoder_multi_subset_scratch_bytes");
        n
    }

    /// `frame_counts[i]` consecutive frames of stream `stream_ids[i]` in ONE call; the same bytes and state as that many
    /// `encode_frames` calls on each listed stream, every other stream untouched.  Device buffers hold the frames packed
    /// row after row in the caller's order: `samples_in` `[total * nf]`, unit v to `buf_out[v * stride ..][.. nbytes]`.
    ///
    /// # Safety
    /// Device pointers valid for the stated extents until the stream has drained.
    pub unsafe fn encode_stream_frames_subset(&mut self, stream_ids: &[i32], frame_counts: &[i32], samples_in: *const i16,
                                              buf_out: *mut u8, nbytes: usize, stride: usize, scratch: DeviceBuf<'_>)
                                              -> Result<(), Lc3EncoderError> {
        assert_eq!(stream_ids.len(), frame_counts.len(), "one frame count per stream id");
        check(sys::lc3b_encode_stream_frames_subset(self.h, stream_ids.as_ptr(), frame_counts.as_ptr(), stream_ids.len() as i32,
                                                    samples_in, buf_out, nbytes as i32, stride, scratch.ptr, scratch.bytes,
                                                    self.stream), "lc3b_encode_stream_frames_subset");
        Ok(())
    }
    pub fn num_streams(&self) -> usize { self.n_streams }
    pub fn samples_per_frame(&self) -> usize { self.nf }
}
impl Drop for Lc3BatchEncoder<'_> {
    fn drop(&mut self) { unsafe { sys::lc3b_encoder_destroy(self.h) } }
}

// --------------------------------------------------------------------------------------------------------------------
// Const-generic twins: the reference offers `Lc3Decoder<'a, const NUM_CHANNELS: usize>` / `Lc3Encoder<..>` for builds
// without an allocator (src/decoder/lc3_decoder.rs:247-310, src/encoder/lc3_encoder.rs:212-304, Cargo.toml:38-40).
// This crate never allocates, so the twins only move the stream count into the type: buffer extents become checkable at
// compile time (`[[u8; NBYTES]; NUM_STREAMS]` style arrays on the caller's side).

/// `Lc3Decoder<'a, NUM_CHANNELS>` of the reference's no-alloc build, batched: `NUM_STREAMS` streams, fixed at compile time.
pub struct Lc3BatchDecoderN<'a, const NUM_STREAMS: usize> {
    inner: Lc3BatchDecoder<'a>,
}

impl<'a, const NUM_STREAMS: usize> Lc3BatchDecoderN<'a, NUM_STREAMS> {
    /// `Lc3Decoder::calc_working_buffer_lengths` (:236) for `NUM_STREAMS` streams.
    pub fn calc_working_buffer_lengths(duration: FrameDuration, freq: SamplingFrequency, max_nbytes: usize) -> usize {
        Lc3BatchDecoder::calc_working_buffer_lengths(NUM_STREAMS, duration, freq, max_nbytes)
    }
    /// `Lc3Decoder::new` (:257 in the no-alloc build)
    pub fn new(duration: FrameDuration, freq: SamplingFrequency, working: DeviceBuf<'a>, max_nbytes: usize, device: i32,
               cuda_stream: *mut c_void) -> Self {
        Self { inner: Lc3BatchDecoder::new(NUM_STREAMS, duration, freq, working, max_nbytes, device, cuda_stream) }
    }
    /// `decode_frame` for all `NUM_STREAMS` streams with HOST arrays whose extents the type system checks:
    /// one `[u8; NBYTES]` frame in and one `[i16; NF]` frame out per stream.
    pub fn decode_frames_host<const NBYTES: usize, const NF: usize>(&mut self, num_bits_per_audio_sample: usize,
                                                                   frames: &[[u8; NBYTES]; NUM_STREAMS],
                                                                   samples_out: &mut [[i16; NF]; NUM_STREAMS])
                                                                   -> Result<(), Lc3DecoderError> {
        assert_eq!(NF, self.inner.samples_per_frame());      // the reference asserts slice lengths the same way
        // pageable host arrays: the copies are synchronous with respect to the host, so the borrows end with the call
        unsafe {
            self.inner.decode_frames(num_bits_per_audio_sample, Residency::Host, frames.as_ptr() as *const u8, ptr::null(),
                                     NBYTES, NBYTES, samples_out.as_mut_ptr() as *mut i16)
        }
    }
    pub fn batch(&mut self) -> &mut Lc3BatchDecoder<'a> { &mut self.inner }
}

/// `Lc3Encoder<'a, NUM_CHANNELS>` of the reference's no-alloc build, batched.
pub struct Lc3BatchEncoderN<'a, const NUM_STREAMS: usize> {
    inner: Lc3BatchEncoder<'a>,
}

impl<'a, const NUM_STREAMS: usize> Lc3BatchEncoderN<'a, NUM_STREAMS> {
    pub fn calc_working_buffer_lengths(duration: FrameDuration, freq: SamplingFrequency, max_nbytes: usize) -> usize {
        Lc3BatchEncoder::calc_working_buffer_lengths(NUM_STREAMS, duration, freq, max_nbytes)
    }
    pub fn new(duration: FrameDuration, freq: SamplingFrequency, working: DeviceBuf<'a>, max_nbytes: usize, device: i32,
               cuda_stream: *mut c_void) -> Self {
        Self { inner: Lc3BatchEncoder::new(NUM_STREAMS, duration, freq, working, max_nbytes, device, cuda_stream) }
    }
    /// `encode_frame` for all `NUM_STREAMS` streams, host arrays: `[i16; NF]` in, `[u8; NBYTES]` out per stream.
    pub fn encode_frames_host<const NBYTES: usize, const NF: usize>(&mut self, samples_in: &[[i16; NF]; NUM_STREAMS],
                                                                   buf_out: &mut [[u8; NBYTES]; NUM_STREAMS])
                                                                   -> Result<(), Lc3EncoderError> {
        assert_eq!(NF, self.inner.samples_per_frame());
        unsafe {
            self.inner.encode_frames(Residency::Host, samples_in.as_ptr() as *const i16, buf_out.as_mut_ptr() as *mut u8,
                                     NBYTES, NBYTES)
        }
    }
    pub fn batch(&mut self) -> &mut Lc3BatchEncoder<'a> { &mut self.inner }
}

// --------------------------------------------------------------------------------------------------------------------
/// Mixed-rate batch (BASELINE config 4): the set of reference decoders a population with different
/// (sampling frequency, frame duration) per stream needs, driven as ONE call.  Rows of every buffer are in BUCKET ORDER:
/// `layout` returns `order[row] = original stream id` and the bucket table.
pub struct Lc3MixedBatchDecoder<'a> {
    h: *mut sys::lc3b_mixed_decoder,
    n_streams: usize,
    stream: *mut c_void,
    _ws: PhantomData<&'a mut [u8]>,
}

/// Bucket table of a mixed-rate population (`lc3b_mixed_decoder_layout`).
pub struct MixedLayout {
    pub buckets: [sys::lc3b_mixed_bucket; sys::LC3B_MIXED_MAX_BUCKETS],
    pub n_buckets: usize,
    /// int16 elements of the dense host PCM buffer `decode_frames_host` fills
    pub host_pcm_elems: usize,
}

impl<'a> Lc3MixedBatchDecoder<'a> {
    /// Row order and buckets for streams with the given per-stream configuration; `order` (optional) receives
    /// `order[row] = original stream id`.
    pub fn layout(freqs: &[SamplingFrequency], durations: &[FrameDuration], order: Option<&mut [i32]>) -> MixedLayout {
        assert_eq!(freqs.len(), durations.len());
        let mut out = MixedLayout { buckets: [sys::lc3b_mixed_bucket::default(); sys::LC3B_MIXED_MAX_BUCKETS], n_buckets: 0, host_pcm_elems: 0 };
        let (mut nb, mut elems) = (0i32, 0u64);
        let order_ptr = match order {
            Some(o) => { assert_eq!(o.len(), freqs.len()); o.as_mut_ptr() }
            None => ptr::null_mut(),
        };
        // the enums are #[repr(i32)] with the C ABI's discriminants
        check(unsafe { sys::lc3b_mixed_decoder_layout(freqs.len() as i32, freqs.as_ptr() as *const i32, durations.as_ptr() as *const i32,
                                                      order_ptr, out.buckets.as_mut_ptr(), &mut nb, &mut elems) },
              "lc3b_mixed_decoder_layout");
        out.n_buckets = nb as usize;
        out.host_pcm_elems = elems as usize;
        out
    }
    /// `calc_working_buffer_lengths` for the whole set.
    pub fn calc_working_buffer_lengths(freqs: &[SamplingFrequency], durations: &[FrameDuration], max_nbytes: usize) -> usize {
        let mut n = 0usize;
        check(unsafe { sys::lc3b_mixed_decoder_workspace_bytes(freqs.len() as i32, freqs.as_ptr() as *const i32,
                                                               durations.as_ptr() as *const i32, max_nbytes as i32, &mut n) },
              "lc3b_mixed_decoder_workspace_bytes");
        n
    }
    /// one `Lc3Decoder::new` per configuration present (src/decoder/lc3_decoder.rs:181), on one borrowed working buffer
    pub fn new(freqs: &[SamplingFrequency], durations: &[FrameDuration], working: DeviceBuf<'a>, max_nbytes: usize,
               device: i32, cuda_stream: *mut c_void) -> Self {
        let mut h = ptr::null_mut();
        check(unsafe { sys::lc3b_mixed_decoder_init(&mut h, freqs.len() as i32, freqs.as_ptr() as *const i32,
                                                    durations.as_ptr() as *const i32, max_nbytes as i32, device, working.ptr,
                                                    working.bytes, cuda_stream) }, "lc3b_mixed_decoder_init");
        Self { h, n_streams: freqs.len(), stream: cuda_stream, _ws: PhantomData }
    }
    /// `decode_frame` for every stream, device buffers, rows in bucket order; `pcm_stride` >= the largest nf.
    ///
    /// # Safety
    /// Device pointers valid for `num_streams` rows until the stream has drained.
    pub unsafe fn decode_frames(&mut self, num_bits_per_audio_sample: usize, frames: *const u8, frame_nbytes: *const i32,
                                nbytes: usize, stride: usize, samples_out: *mut i16, pcm_stride: usize, status_out: *mut i32)
                                -> Result<(), Lc3DecoderError> {
        match sys::lc3b_mixed_decode_frames(self.h, num_bits_per_audio_sample as i32, frames, frame_nbytes, nbytes as i32, stride,
                                            samples_out, pcm_stride, status_out, self.stream) {
            sys::LC3B_OK => Ok(()),
            sys::LC3B_ERR_BITS_PER_SAMPLE => Err(Lc3DecoderError::Only16BitsPerAudioSampleSupported),
            rc => { check(rc, "lc3b_mixed_decode_frames"); unreachable!() }
        }
    }
    /// Same with host buffers; `samples_out` is the dense per-bucket buffer of `MixedLayout::host_pcm_elems` elements.
    ///
    /// # Safety
    /// Host pointers (pinned for asynchronous copies) valid until the stream has drained.
    pub unsafe fn decode_frames_host(&mut self, num_bits_per_audio_sample: usize, frames: *const u8, frame_nbytes: *const i32,
                                     nbytes: usize, stride: usize, samples_out: *mut i16, status_out: *mut i32)
                                     -> Result<(), Lc3DecoderError> {
        match sys::lc3b_mixed_decode_frames_host(self.h, num_bits_per_audio_sample as i32, frames, frame_nbytes, nbytes as i32, stride,
                                                 samples_out, status_out, self.stream) {
            sys::LC3B_OK => Ok(()),
            sys::LC3B_ERR_BITS_PER_SAMPLE => Err(Lc3DecoderError::Only16BitsPerAudioSampleSupported),
            rc => { check(rc, "lc3b_mixed_decode_frames_host"); unreachable!() }
        }
    }
    pub fn set_host_pipelining(&mut self, on: bool) {
        check(unsafe { sys::lc3b_mixed_decoder_set_host_pipelining(self.h, on as i32) }, "lc3b_mixed_decoder_set_host_pipelining");
    }
    pub fn host_fence(&mut self) {
        check(unsafe { sys::lc3b_mixed_decoder_host_fence(self.h, self.stream) }, "lc3b_mixed_decoder_host_fence");
    }
    pub fn num_streams(&self) -> usize { self.n_streams }
}
impl Drop for Lc3MixedBatchDecoder<'_> {
    fn drop(&mut self) { unsafe { sys::lc3b_mixed_decoder_destroy(self.h) } }
}

// --------------------------------------------------------------------------------------------------------------------
/// One batch over the GPUs of a box (BASELINE config 5): streams are independent (src/decoder/lc3_decoder.rs:62-69), so
/// stream s goes to shard floor(s * G / N); one host thread, CUDA stream and device workspace per GPU, owned by the handle.
pub struct Lc3ShardedBatchDecoder {
    h: *mut sys::lc3b_sharded_decoder,
    n_streams: usize,
}

impl Lc3ShardedBatchDecoder {
    /// `devices`: CUDA device indices, one shard each.
    pub fn new(num_streams: usize, duration: FrameDuration, freq: SamplingFrequency, max_nbytes: usize, devices: &[i32]) -> Self {
        let mut h = ptr::null_mut();
        check(unsafe { sys::lc3b_sharded_decoder_create(&mut h, num_streams as i32, duration as i32, freq as i32, max_nbytes as i32,
                                                        devices.as_ptr(), devices.len() as i32) }, "lc3b_sharded_decoder_create");
        Self { h, n_streams: num_streams }
    }
    /// (device, first stream, stream count) of shard `g`.
    pub fn shard(&self, g: usize) -> (i32, usize, usize) {
        let (mut d, mut f, mut n) = (0i32, 0i32, 0i32);
        check(unsafe { sys::lc3b_sharded_decoder_shard(self.h, g as i32, &mut d, &mut f, &mut n) }, "lc3b_sharded_decoder_shard");
        (d, f as usize, n as usize)
    }
    pub fn num_shards(&self) -> usize { unsafe { sys::lc3b_sharded_decoder_n_shards(self.h) as usize } }
    /// `decode_frame` for every stream of the batch; host (pinned) buffers for ALL streams.  Returns once every GPU's
    /// thread has the call; `wait` joins.
    ///
    /// # Safety
    /// The host buffers must stay valid and untouched until `wait` returns.
    pub unsafe fn decode_frames_host(&mut self, num_bits_per_audio_sample: usize, frames: *const u8, frame_nbytes: *const i32,
                                     nbytes: usize, stride: usize, samples_out: *mut i16, pcm_stride: usize, status_out: *mut i32)
                                     -> Result<(), Lc3DecoderError> {
        match sys::lc3b_sharded_decode_frames_host(self.h, num_bits_per_audio_sample as i32, frames, frame_nbytes, nbytes as i32,
                                                   stride, samples_out, pcm_stride, status_out) {
            sys::LC3B_OK => Ok(()),
            sys::LC3B_ERR_BITS_PER_SAMPLE => Err(Lc3DecoderError::Only16BitsPerAudioSampleSupported),
            rc => { check(rc, "lc3b_sharded_decode_frames_host"); unreachable!() }
        }
    }
    /// Joins every outstanding call on every GPU; outputs are valid afterwards.
    pub fn wait(&mut self) { check(unsafe { sys::lc3b_sharded_decoder_wait(self.h) }, "lc3b_sharded_decoder_wait"); }
    pub fn num_streams(&self) -> usize { self.n_streams }
}
impl Drop for Lc3ShardedBatchDecoder {
    fn drop(&mut self) { unsafe { sys::lc3b_sharded_decoder_destroy(self.h) } }
}

/// The encoder counterpart of `Lc3ShardedBatchDecoder` (src/encoder/lc3_encoder.rs:42-60: channels are independent).
pub struct Lc3ShardedBatchEncoder {
    h: *mut sys::lc3b_sharded_encoder,
    n_streams: usize,
}

impl Lc3ShardedBatchEncoder {
    pub fn new(num_streams: usize, duration: FrameDuration, freq: SamplingFrequency, max_nbytes: usize, devices: &[i32]) -> Self {
        let mut h = ptr::null_mut();
        check(unsafe { sys::lc3b_sharded_encoder_create(&mut h, num_streams as i32, duration as i32, freq as i32, max_nbytes as i32,
                                                        devices.as_ptr(), devices.len() as i32) }, "lc3b_sharded_encoder_create");
        Self { h, n_streams: num_streams }
    }
    /// # Safety
    /// The host buffers must stay valid and untouched until `wait` returns.
    pub unsafe fn encode_frames_host(&mut self, samples_in: *const i16, pcm_stride: usize, buf_out: *mut u8, nbytes: usize,
                                     stride: usize) -> Result<(), Lc3EncoderError> {
        check(sys::lc3b_sharded_encode_frames_host(self.h, samples_in, pcm_stride, buf_out, nbytes as i32, stride),
              "lc3b_sharded_encode_frames_host");
        Ok(())
    }
    pub fn wait(&mut self) { check(unsafe { sys::lc3b_sharded_encoder_wait(self.h) }, "lc3b_sharded_encoder_wait"); }
    pub fn num_streams(&self) -> usize { self.n_streams }
}
impl Drop for Lc3ShardedBatchEncoder {
    fn drop(&mut self) { unsafe { sys::lc3b_sharded_encoder_destroy(self.h) } }
}
