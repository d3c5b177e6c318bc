// lc3b - C++ host-side mirror of the reference's operator interface for the hot path.
//
// The reference (ninjasource/lc3-codec) is Rust; this image has no Rust toolchain, so the host side above the C ABI
// (include/lc3b.h) is written in C++ with the reference's names, argument meaning and error behaviour:
//
//   reference (file:line)                                          here
//   Lc3Decoder::calc_working_buffer_lengths  lc3_decoder.rs:236     lc3b::Lc3BatchDecoder::calc_working_buffer_lengths
//   Lc3Decoder::new                          lc3_decoder.rs:181     lc3b::Lc3BatchDecoder::Lc3BatchDecoder
//   Lc3Decoder::decode_frame                 lc3_decoder.rs:217     lc3b::Lc3BatchDecoder::decode_frames (one call = every stream)
//   Lc3DecoderError                          lc3_decoder.rs:36      lc3b::Lc3DecoderError
//   Lc3Encoder::{calc_working_buffer_lengths,new,encode_frame}  lc3_encoder.rs:194,:117,:175   lc3b::Lc3BatchEncoder
//   Lc3Config::new                           config.rs:42           lc3b::Lc3Config
//   one Lc3Decoder per (duration, frequency) lc3_decoder.rs:181     lc3b::Lc3MixedBatchDecoder (mixed-rate population, one call)
//   independent channels                     lc3_decoder.rs:62-69   lc3b::Lc3ShardedBatchDecoder / Lc3ShardedBatchEncoder (one batch, many GPUs)
//
// Preallocated-buffer style as in the reference: the caller asks for the working-buffer size, allocates it (device
// memory, 256-byte aligned) and lends it to the constructor; nothing is allocated on the device afterwards.
// Error behaviour: the one error the reference returns comes back as a value (Result); misuse the reference answers
// with a panic (bad sizes, 8 kHz encoder) throws std::logic_error; CUDA failures throw std::runtime_error.
// Header-only; link with -llc3b.
#pragma once
#include <cstddef>
#include <cstdint>
#include <optional>
#include <stdexcept>
#include <string>
#include <vector>

#include "lc3b.h"

namespace lc3b {

enum class SamplingFrequency : int { Hz8000 = LC3B_HZ8000, Hz16000, Hz24000, Hz32000, Hz44100, Hz48000 };   // config.rs:2
enum class FrameDuration : int { SevenPointFiveMs = LC3B_7P5MS, TenMs = LC3B_10MS };                          // config.rs:12

// Lc3DecoderError (lc3_decoder.rs:36-41).  Bitstream errors never surface: they are concealed (:138-141).
enum class Lc3DecoderError { Only16BitsPerAudioSampleSupported };
// Result<(), E>: empty optional == Ok(())
template <class E>
using Result = std::optional<E>;
// Lc3EncoderError is an empty enum in the reference (lc3_encoder.rs:30): encode_frame cannot fail.
enum class Lc3EncoderError {};

namespace detail {
inline void check(int rc, const char* what) {
    if (rc == LC3B_OK) return;
    const std::string msg = std::string("lc3b: ") + what + " failed with status " + std::to_string(rc);
    if (rc == LC3B_ERR_INVALID_ARG) throw std::logic_error(msg + " (the reference panics here)");
    throw std::runtime_error(msg + " (cuda error " + std::to_string(lc3b_last_cuda_error()) + ")");
}
}  // namespace detail

// Lc3Config (config.rs:18-39)
struct Lc3Config {
    int fs_ind, fs, ne, nb, nf, z;
    FrameDuration n_ms;
    Lc3Config(SamplingFrequency f, FrameDuration d) {
        lc3b_config c;
        detail::check(lc3b_config_new((int)f, (int)d, &c), "lc3b_config_new");
        fs_ind = c.fs_ind; fs = c.fs; ne = c.ne; nb = c.nb; nf = c.nf; z = c.z; n_ms = d;
    }
};

// Where a call's I/O buffers live: device pointers (no copies, asynchronous) or host pointers (the library stages
// the transfers; asynchronous when pinned).
enum class Residency { Device, Host };

class Lc3BatchDecoder {
  public:
    // Lc3Decoder::calc_working_buffer_lengths: bytes of device working memory for `num_streams` channels
    static size_t calc_working_buffer_lengths(size_t num_streams, FrameDuration d, SamplingFrequency f, size_t max_nbytes) {
        size_t n = 0;
        detail::check(lc3b_decoder_workspace_bytes((int)num_streams, (int)d, (int)f, (int)max_nbytes, &n), "lc3b_decoder_workspace_bytes");
        return n;
    }
    // Lc3Decoder::new: borrows `working` (device memory) for the lifetime of the object; state starts zeroed
    Lc3BatchDecoder(size_t num_streams, FrameDuration d, SamplingFrequency f, void* working, size_t working_bytes,
                    size_t max_nbytes, int device = 0, void* cuda_stream = nullptr)
        : config(f, d), num_streams_(num_streams), stream_(cuda_stream) {
        detail::check(lc3b_decoder_init(&h_, (int)num_streams, (int)d, (int)f, (int)max_nbytes, device, working, working_bytes, cuda_stream),
                      "lc3b_decoder_init");
    }
    Lc3BatchDecoder(const Lc3BatchDecoder&) = delete;
    Lc3BatchDecoder& operator=(const Lc3BatchDecoder&) = delete;
    ~Lc3BatchDecoder() { lc3b_decoder_destroy(h_); }

    // decode_frame for every stream: frames[s * frame_stride .. + nbytes] -> samples_out[s * nf .. (s+1) * nf].
    // frame_nbytes (nullable, same residency): per-stream buf_in.len(); 0 = lost frame, concealed like the reference.
    Result<Lc3DecoderError> decode_frames(size_t num_bits_per_audio_sample, Residency where, const uint8_t* frames,
                                          size_t nbytes, size_t frame_stride, int16_t* samples_out,
                                          const int32_t* frame_nbytes = nullptr, int32_t* status_out = nullptr) {
        auto fn = where == Residency::Device ? lc3b_decode_frames : lc3b_decode_frames_host;
        const int rc = fn(h_, (int)num_bits_per_audio_sample, frames, frame_nbytes, (int)nbytes, frame_stride, samples_out,
                          (size_t)config.nf, status_out, stream_);
        if (rc == LC3B_ERR_BITS_PER_SAMPLE) return Lc3DecoderError::Only16BitsPerAudioSampleSupported;
        detail::check(rc, "lc3b_decode_frames");
        return std::nullopt;
    }
    // decode_frame (lc3_decoder.rs:217) for the listed streams only, every other stream untouched.  Row i of the device
    // buffers (frames, samples_out, frame_nbytes, status_out) belongs to stream stream_ids[i]; stream_ids is a host array of
    // n_rows distinct ids in [0, num_streams), only read during the call (a bad list throws, like the reference's panic).
    Result<Lc3DecoderError> decode_frames_subset(size_t num_bits_per_audio_sample, const int32_t* stream_ids, size_t n_rows,
                                                 const uint8_t* frames, size_t nbytes, size_t frame_stride, int16_t* samples_out,
                                                 const int32_t* frame_nbytes = nullptr, int32_t* status_out = nullptr) {
        const int rc = lc3b_decode_frames_subset(h_, (int)num_bits_per_audio_sample, stream_ids, (int)n_rows, frames, frame_nbytes,
                                                 (int)nbytes, frame_stride, samples_out, (size_t)config.nf, status_out, stream_);
        if (rc == LC3B_ERR_BITS_PER_SAMPLE) return Lc3DecoderError::Only16BitsPerAudioSampleSupported;
        detail::check(rc, "lc3b_decode_frames_subset");
        return std::nullopt;
    }
    // the listed streams start over with the state Lc3Decoder::new gives a channel; no other stream is touched
    void reset_streams(const int32_t* stream_ids, size_t n) {
        detail::check(lc3b_decoder_reset_streams(h_, stream_ids, (int)n, stream_), "lc3b_decoder_reset_streams");
    }
    // Time-parallel decode (SURVEY.md 8f-1): n_frames consecutive frames of every stream in one call; equivalent to
    // n_frames decode_frames calls (same PCM, same state afterwards).  Device buffers: frames [num_streams][n_frames][nbytes],
    // samples_out [num_streams][n_frames * nf], scratch >= multi_scratch_bytes(n_frames) bytes (caller-owned).
    size_t multi_scratch_bytes(size_t n_frames) const {
        size_t n = 0;
        detail::check(lc3b_decoder_multi_scratch_bytes(h_, (int)n_frames, &n), "lc3b_decoder_multi_scratch_bytes");
        return n;
    }
    Result<Lc3DecoderError> decode_stream_frames(size_t num_bits_per_audio_sample, const uint8_t* frames, size_t nbytes,
                                                 size_t n_frames, int16_t* samples_out, void* scratch, size_t scratch_bytes,
                                                 const int32_t* frame_nbytes = nullptr, int32_t* status_out = nullptr) {
        const int rc = lc3b_decode_stream_frames(h_, (int)num_bits_per_audio_sample, frames, frame_nbytes, (int)nbytes, nbytes,
                                                 (int)n_frames, samples_out, status_out, scratch, scratch_bytes, stream_);
        if (rc == LC3B_ERR_BITS_PER_SAMPLE) return Lc3DecoderError::Only16BitsPerAudioSampleSupported;
        detail::check(rc, "lc3b_decode_stream_frames");
        return std::nullopt;
    }
    // Ragged time-parallel decode: frame_counts[i] consecutive frames of stream stream_ids[i] (host arrays of n_rows, ids
    // as in decode_frames_subset, counts >= 0); equivalent to that many decode_frames calls on each listed stream.  Units are
    // packed row after row in the caller's order: device frames [total][nbytes], samples_out [total * nf], frame_nbytes /
    // status_out [total]; scratch >= multi_subset_scratch_bytes(n_rows, total) bytes (caller-owned).
    size_t multi_subset_scratch_bytes(size_t n_rows, long long total_frames) const {
        size_t n = 0;
        detail::check(lc3b_decoder_multi_subset_scratch_bytes(h_, (int)n_rows, total_frames, &n), "lc3b_decoder_multi_subset_scratch_bytes");
        return n;
    }
    Result<Lc3DecoderError> decode_stream_frames_subset(size_t num_bits_per_audio_sample, const int32_t* stream_ids,
                                                        const int32_t* frame_counts, size_t n_rows, const uint8_t* frames,
                                                        size_t nbytes, int16_t* samples_out, void* scratch, size_t scratch_bytes,
                                                        const int32_t* frame_nbytes = nullptr, int32_t* status_out = nullptr) {
        const int rc = lc3b_decode_stream_frames_subset(h_, (int)num_bits_per_audio_sample, stream_ids, frame_counts, (int)n_rows,
                                                        frames, frame_nbytes, (int)nbytes, nbytes, samples_out, status_out, scratch,
                                                        scratch_bytes, stream_);
        if (rc == LC3B_ERR_BITS_PER_SAMPLE) return Lc3DecoderError::Only16BitsPerAudioSampleSupported;
        detail::check(rc, "lc3b_decode_stream_frames_subset");
        return std::nullopt;
    }
    // extension: issue every call as one cached CUDA graph (true) or one launch per kernel (false); same results
    void set_graph_mode(bool on) { detail::check(lc3b_decoder_set_graph_mode(h_, on ? 1 : 0), "lc3b_decoder_set_graph_mode"); }
    // extension: cut every call into k independent sub-batches whose kernels overlap (0 = by batch size, 1, 2, 4); same results
    void set_split(int k) { detail::check(lc3b_decoder_set_split(h_, k), "lc3b_decoder_set_split"); }
    // extension: overlap the PCM read-back of call i with the kernels of call i+1 (host residency)
    void set_host_pipelining(bool on) { detail::check(lc3b_decoder_set_host_pipelining(h_, on ? 1 : 0), "lc3b_decoder_set_host_pipelining"); }
    void host_fence() { detail::check(lc3b_decoder_host_fence(h_, stream_), "lc3b_decoder_host_fence"); }

    size_t num_streams() const { return num_streams_; }
    lc3b_decoder* handle() { return h_; }
    const Lc3Config config;

  private:
    lc3b_decoder* h_ = nullptr;
    size_t num_streams_;
    void* stream_;
};

class Lc3BatchEncoder {
  public:
    // Lc3Encoder::calc_working_buffer_lengths (lc3_encoder.rs:194).  8 kHz: std::logic_error, the reference's
    // Lc3Encoder::new panics there (bandwidth_detector.rs:42-56).
    static size_t calc_working_buffer_lengths(size_t num_streams, FrameDuration d, SamplingFrequency f, size_t max_nbytes) {
        size_t n = 0;
        detail::check(lc3b_encoder_workspace_bytes((int)num_streams, (int)d, (int)f, (int)max_nbytes, &n), "lc3b_encoder_workspace_bytes");
        return n;
    }
    // Lc3Encoder::new (lc3_encoder.rs:117)
    Lc3BatchEncoder(size_t num_streams, FrameDuration d, SamplingFrequency f, void* working, size_t working_bytes,
                    size_t max_nbytes, int device = 0, void* cuda_stream = nullptr)
        : config(f, d), num_streams_(num_streams), stream_(cuda_stream) {
        detail::check(lc3b_encoder_init(&h_, (int)num_streams, (int)d, (int)f, (int)max_nbytes, device, working, working_bytes, cuda_stream),
                      "lc3b_encoder_init");
    }
    Lc3BatchEncoder(const Lc3BatchEncoder&) = delete;
    Lc3BatchEncoder& operator=(const Lc3BatchEncoder&) = delete;
    ~Lc3BatchEncoder() { lc3b_encoder_destroy(h_); }

    // encode_frame (lc3_encoder.rs:175) for every stream: samples_in[s * nf ..] -> buf_out[s * frame_stride .. + nbytes]
    Result<Lc3EncoderError> encode_frames(Residency where, const int16_t* samples_in, uint8_t* buf_out, size_t nbytes,
                                          size_t frame_stride) {
        auto fn = where == Residency::Device ? lc3b_encode_frames : lc3b_encode_frames_host;
        detail::check(fn(h_, samples_in, (size_t)config.nf, buf_out, (int)nbytes, frame_stride, stream_), "lc3b_encode_frames");
        return std::nullopt;
    }
    // encode_frame (lc3_encoder.rs:175) for the listed streams only: row i of the device buffers belongs to stream
    // stream_ids[i] (host array of n_rows distinct ids, only read during the call)
    Result<Lc3EncoderError> encode_frames_subset(const int32_t* stream_ids, size_t n_rows, const int16_t* samples_in, uint8_t* buf_out,
                                                 size_t nbytes, size_t frame_stride) {
        detail::check(lc3b_encode_frames_subset(h_, stream_ids, (int)n_rows, samples_in, (size_t)config.nf, buf_out, (int)nbytes,
                                                frame_stride, stream_),
                      "lc3b_encode_frames_subset");
        return std::nullopt;
    }
    // the listed streams start over with the state Lc3Encoder::new gives a channel; no other stream is touched
    void reset_streams(const int32_t* stream_ids, size_t n) {
        detail::check(lc3b_encoder_reset_streams(h_, stream_ids, (int)n, stream_), "lc3b_encoder_reset_streams");
    }
    // Time-parallel encode: n_frames consecutive frames of every stream in one call; equivalent to n_frames encode_frames
    // calls (same bytes, same state afterwards).  Device buffers: samples_in [num_streams][n_frames * nf], buf_out frame f of
    // stream s at (s * n_frames + f) * frame_stride, scratch >= multi_scratch_bytes(n_frames) bytes (caller-owned).
    size_t multi_scratch_bytes(size_t n_frames) const {
        size_t n = 0;
        detail::check(lc3b_encoder_multi_scratch_bytes(h_, (int)n_frames, &n), "lc3b_encoder_multi_scratch_bytes");
        return n;
    }
    Result<Lc3EncoderError> encode_stream_frames(const int16_t* samples_in, size_t n_frames, uint8_t* buf_out, size_t nbytes,
                                                 size_t frame_stride, void* scratch, size_t scratch_bytes) {
        detail::check(lc3b_encode_stream_frames(h_, samples_in, (int)n_frames, buf_out, (int)nbytes, frame_stride, scratch,
                                                scratch_bytes, stream_),
                      "lc3b_encode_stream_frames");
        return std::nullopt;
    }
    // Ragged time-parallel encode: frame_counts[i] consecutive frames of stream stream_ids[i] (host arrays of n_rows);
    // equivalent to that many encode_frames calls on each listed stream.  Units packed row after row in the caller's
    // order: samples_in [total * nf], buf_out unit v at v * frame_stride; scratch >= multi_subset_scratch_bytes(n_rows, total).
    size_t multi_subset_scratch_bytes(size_t n_rows, long long total_frames) const {
        size_t n = 0;
        detail::check(lc3b_encoder_multi_subset_scratch_bytes(h_, (int)n_rows, total_frames, &n), "lc3b_encoder_multi_subset_scratch_bytes");
        return n;
    }
    Result<Lc3EncoderError> encode_stream_frames_subset(const int32_t* stream_ids, const int32_t* frame_counts, size_t n_rows,
                                                        const int16_t* samples_in, uint8_t* buf_out, size_t nbytes, size_t frame_stride,
                                                        void* scratch, size_t scratch_bytes) {
        detail::check(lc3b_encode_stream_frames_subset(h_, stream_ids, frame_counts, (int)n_rows, samples_in, buf_out, (int)nbytes,
                                                       frame_stride, scratch, scratch_bytes, stream_),
                      "lc3b_encode_stream_frames_subset");
        return std::nullopt;
    }
    void set_host_pipelining(bool on) { detail::check(lc3b_encoder_set_host_pipelining(h_, on ? 1 : 0), "lc3b_encoder_set_host_pipelining"); }

    size_t num_streams() const { return num_streams_; }
    lc3b_encoder* handle() { return h_; }
    const Lc3Config config;

  private:
    lc3b_encoder* h_ = nullptr;
    size_t num_streams_;
    void* stream_;
};

// Mixed-rate batch (BASELINE config 4).  The reference's Lc3Decoder::new takes ONE frame duration and ONE sampling
// frequency for all channels (lc3_decoder.rs:181), so a population with per-stream configurations is a set of
// decoders; this is that set behind one call.  Rows of every buffer are in BUCKET ORDER: order()[row] = original
// stream id, buckets() gives each configuration's row range (include/lc3b.h, lc3b_mixed_*).
class Lc3MixedBatchDecoder {
  public:
    struct Layout {
        std::vector<int32_t> order;
        std::vector<lc3b_mixed_bucket> buckets;
        size_t host_pcm_elems = 0;
    };
    static Layout layout(const std::vector<SamplingFrequency>& f, const std::vector<FrameDuration>& d) {
        if (f.size() != d.size()) throw std::logic_error("lc3b: one frequency and one duration per stream");
        Layout L;
        L.order.resize(f.size());
        L.buckets.resize(LC3B_MIXED_MAX_BUCKETS);
        int32_t nb = 0;
        uint64_t elems = 0;
        detail::check(lc3b_mixed_decoder_layout((int)f.size(), (const int32_t*)f.data(), (const int32_t*)d.data(), L.order.data(),
                                                L.buckets.data(), &nb, &elems), "lc3b_mixed_decoder_layout");
        L.buckets.resize((size_t)nb);
        L.host_pcm_elems = (size_t)elems;
        return L;
    }
    static size_t calc_working_buffer_lengths(const std::vector<SamplingFrequency>& f, const std::vector<FrameDuration>& d,
                                              size_t max_nbytes) {
        size_t n = 0;
        detail::check(lc3b_mixed_decoder_workspace_bytes((int)f.size(), (const int32_t*)f.data(), (const int32_t*)d.data(),
                                                         (int)max_nbytes, &n), "lc3b_mixed_decoder_workspace_bytes");
        return n;
    }
    Lc3MixedBatchDecoder(const std::vector<SamplingFrequency>& f, const std::vector<FrameDuration>& d, void* working,
                         size_t working_bytes, size_t max_nbytes, int device = 0, void* cuda_stream = nullptr)
        : layout_(layout(f, d)), stream_(cuda_stream) {
        detail::check(lc3b_mixed_decoder_init(&h_, (int)f.size(), (const int32_t*)f.data(), (const int32_t*)d.data(), (int)max_nbytes,
                                              device, working, working_bytes, cuda_stream), "lc3b_mixed_decoder_init");
    }
    Lc3MixedBatchDecoder(const Lc3MixedBatchDecoder&) = delete;
    Lc3MixedBatchDecoder& operator=(const Lc3MixedBatchDecoder&) = delete;
    ~Lc3MixedBatchDecoder() { lc3b_mixed_decoder_destroy(h_); }

    // decode_frame for every stream.  Device residency: samples_out rows share the pitch pcm_stride (>= largest nf).
    // Host residency: samples_out is dense per bucket (Layout::host_pcm_elems int16, bucket b at host_pcm_offset); pcm_stride unused.
    Result<Lc3DecoderError> decode_frames(size_t num_bits_per_audio_sample, Residency where, const uint8_t* frames,
                                          const int32_t* frame_nbytes, size_t nbytes, size_t frame_stride, int16_t* samples_out,
                                          size_t pcm_stride, int32_t* status_out = nullptr) {
        const int rc = where == Residency::Device
                           ? lc3b_mixed_decode_frames(h_, (int)num_bits_per_audio_sample, frames, frame_nbytes, (int)nbytes, frame_stride,
                                                      samples_out, pcm_stride, status_out, stream_)
                           : lc3b_mixed_decode_frames_host(h_, (int)num_bits_per_audio_sample, frames, frame_nbytes, (int)nbytes,
                                                           frame_stride, samples_out, status_out, stream_);
        if (rc == LC3B_ERR_BITS_PER_SAMPLE) return Lc3DecoderError::Only16BitsPerAudioSampleSupported;
        detail::check(rc, "lc3b_mixed_decode_frames");
        return std::nullopt;
    }
    void set_host_pipelining(bool on) { detail::check(lc3b_mixed_decoder_set_host_pipelining(h_, on ? 1 : 0), "lc3b_mixed_decoder_set_host_pipelining"); }
    void host_fence() { detail::check(lc3b_mixed_decoder_host_fence(h_, stream_), "lc3b_mixed_decoder_host_fence"); }
    const std::vector<int32_t>& order() const { return layout_.order; }
    const std::vector<lc3b_mixed_bucket>& buckets() const { return layout_.buckets; }
    size_t host_pcm_elems() const { return layout_.host_pcm_elems; }

  private:
    Layout layout_;
    lc3b_mixed_decoder* h_ = nullptr;
    void* stream_;
};

// One batch over several GPUs (BASELINE config 5): channels never interact (lc3_decoder.rs:62-69, lc3_encoder.rs:42-60),
// so stream s goes to shard floor(s * G / N) and nothing is exchanged.  The handle owns a device workspace, a CUDA stream and
// a host thread per GPU; calls take HOST buffers (pin them) for the whole batch and return at once, wait() joins.
class Lc3ShardedBatchDecoder {
  public:
    Lc3ShardedBatchDecoder(size_t num_streams, FrameDuration d, SamplingFrequency f, size_t max_nbytes, const std::vector<int>& devices)
        : config(f, d) {
        detail::check(lc3b_sharded_decoder_create(&h_, (int)num_streams, (int)d, (int)f, (int)max_nbytes, devices.data(), (int)devices.size()),
                      "lc3b_sharded_decoder_create");
    }
    Lc3ShardedBatchDecoder(const Lc3ShardedBatchDecoder&) = delete;
    Lc3ShardedBatchDecoder& operator=(const Lc3ShardedBatchDecoder&) = delete;
    ~Lc3ShardedBatchDecoder() { lc3b_sharded_decoder_destroy(h_); }
    Result<Lc3DecoderError> decode_frames(size_t num_bits_per_audio_sample, const uint8_t* frames, size_t nbytes, size_t frame_stride,
                                          int16_t* samples_out, const int32_t* frame_nbytes = nullptr, int32_t* status_out = nullptr) {
        const int rc = lc3b_sharded_decode_frames_host(h_, (int)num_bits_per_audio_sample, frames, frame_nbytes, (int)nbytes, frame_stride,
                                                       samples_out, (size_t)config.nf, status_out);
        if (rc == LC3B_ERR_BITS_PER_SAMPLE) return Lc3DecoderError::Only16BitsPerAudioSampleSupported;
        detail::check(rc, "lc3b_sharded_decode_frames_host");
        return std::nullopt;
    }
    void wait() { detail::check(lc3b_sharded_decoder_wait(h_), "lc3b_sharded_decoder_wait"); }
    int num_shards() const { return lc3b_sharded_decoder_n_shards(h_); }
    const Lc3Config config;

  private:
    lc3b_sharded_decoder* h_ = nullptr;
};

class Lc3ShardedBatchEncoder {
  public:
    Lc3ShardedBatchEncoder(size_t num_streams, FrameDuration d, SamplingFrequency f, size_t max_nbytes, const std::vector<int>& devices)
        : config(f, d) {
        detail::check(lc3b_sharded_encoder_create(&h_, (int)num_streams, (int)d, (int)f, (int)max_nbytes, devices.data(), (int)devices.size()),
                      "lc3b_sharded_encoder_create");
    }
    Lc3ShardedBatchEncoder(const Lc3ShardedBatchEncoder&) = delete;
    Lc3ShardedBatchEncoder& operator=(const Lc3ShardedBatchEncoder&) = delete;
    ~Lc3ShardedBatchEncoder() { lc3b_sharded_encoder_destroy(h_); }
    Result<Lc3EncoderError> encode_frames(const int16_t* samples_in, uint8_t* buf_out, size_t nbytes, size_t frame_stride) {
        detail::check(lc3b_sharded_encode_frames_host(h_, samples_in, (size_t)config.nf, buf_out, (int)nbytes, frame_stride),
                      "lc3b_sharded_encode_frames_host");
        return std::nullopt;
    }
    void wait() { detail::check(lc3b_sharded_encoder_wait(h_), "lc3b_sharded_encoder_wait"); }
    int num_shards() const { return lc3b_sharded_encoder_n_shards(h_); }
    const Lc3Config config;

  private:
    lc3b_sharded_encoder* h_ = nullptr;
};

}  // namespace lc3b
