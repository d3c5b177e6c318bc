/* lc3b - batched LC3 codec engine for NVIDIA B200 (sm_100a): public C ABI.
 *
 * Drop-in boundary for ONE path of ninjasource/lc3-codec: Lc3Decoder::decode_frame /
 * Lc3Encoder::encode_frame, batched over many independent streams ("stream" plays the
 * role of the reference's channel_index).  The reference has no FFI layer; each entry
 * point below names the inherent method it replaces (paths relative to the reference
 * root, SURVEY.md section 8b).  Plain pointers and sizes only - no C++/torch types.
 *
 * Ownership mirrors the reference's preallocated-buffer style: the caller allocates the
 * device workspace (size from *_workspace_bytes) and all I/O buffers; the library
 * allocates nothing on the device after init and never frees caller memory.
 *
 * Threading: a handle is not thread-safe (the reference takes &mut self); calls are
 * asynchronous on the caller's CUDA stream and ordered within it; frames of a stream
 * must be submitted in order; different handles are independent.
 *
 * There is no CPU fallback: every entry point that does work requires a CUDA device.
 */
#ifndef LC3B_H
#define LC3B_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* status codes (never unwinds across the boundary) */
enum {
    LC3B_OK = 0,
    LC3B_ERR_BITS_PER_SAMPLE = 1, /* Lc3DecoderError::Only16BitsPerAudioSampleSupported, src/decoder/lc3_decoder.rs:80 */
    LC3B_ERR_INVALID_ARG = 2,     /* where the reference panics (bad channel index :228, wrong slice length asserts) */
    LC3B_ERR_CUDA = 3,            /* a CUDA runtime call failed; lc3b_last_cuda_error() has the code */
    LC3B_ERR_WORKSPACE = 4        /* workspace too small or misaligned */
};

/* SamplingFrequency, src/common/config.rs:2 (44.1 kHz shares every size with 48 kHz, :48-49) */
enum { LC3B_HZ8000 = 0, LC3B_HZ16000 = 1, LC3B_HZ24000 = 2, LC3B_HZ32000 = 3, LC3B_HZ44100 = 4, LC3B_HZ48000 = 5 };
/* FrameDuration, src/common/config.rs:12 */
enum { LC3B_7P5MS = 0, LC3B_10MS = 1 };

/* Lc3Config, src/common/config.rs:18-39 */
typedef struct lc3b_config {
    int32_t fs_ind, fs, ne, nb, nf, z, n_ms;
} lc3b_config;

/* Lc3Config::new, src/common/config.rs:42.  Returns LC3B_ERR_INVALID_ARG for unknown enums. */
int lc3b_config_new(int sampling_frequency, int frame_duration, lc3b_config* out);

int lc3b_last_cuda_error(void);
const char* lc3b_version(void);

/* ------------------------------------------------------------------ decoder */
typedef struct lc3b_decoder lc3b_decoder;

/* Lc3Decoder::calc_working_buffer_lengths, src/decoder/lc3_decoder.rs:236.
 * max_nbytes: largest frame length (bytes) that will ever be submitted (<= 400). */
int lc3b_decoder_workspace_bytes(int n_streams, int frame_duration, int sampling_frequency, int max_nbytes,
                                 size_t* device_bytes);

/* Lc3Decoder::new, src/decoder/lc3_decoder.rs:181.  `dev_workspace` is device memory of at least
 * `device_bytes`, 256-byte aligned; it is zero-filled and initialised here (plc_seed = 24607, alpha = 1,
 * packet_loss_concealment.rs:31-33) on `cuda_stream`. */
int lc3b_decoder_init(lc3b_decoder** out, int n_streams, int frame_duration, int sampling_frequency, int max_nbytes,
                      int device, void* dev_workspace, size_t workspace_bytes, void* cuda_stream);

/* One Lc3Decoder::decode_frame (src/decoder/lc3_decoder.rs:217) per stream, for all streams of the handle.
 *   frames        device, stream-major: frame of stream s at frames + s*frame_stride
 *   frame_nbytes  device int32[n_streams] or NULL.  NULL: every frame is `nbytes` long.  Otherwise the per-stream
 *                 `buf_in.len()`; 0 hands the decoder an empty slice, which the reference conceals (:138-141).
 *   nbytes        frame length when frame_nbytes is NULL, and upper bound otherwise (<= max_nbytes, <= frame_stride)
 *   pcm_out       device, int16, stream s at pcm_out + s*pcm_stride (elements); nf samples are written
 *   status_out    device int32[n_streams] or NULL: 0 = decoded, 1 = concealed (an extension: the reference hides it)
 * Returns LC3B_ERR_BITS_PER_SAMPLE when bits_per_sample != 16, like the reference; nothing is launched then. */
int lc3b_decode_frames(lc3b_decoder* h, int bits_per_sample, const uint8_t* frames, const int32_t* frame_nbytes,
                       int nbytes, size_t frame_stride, int16_t* pcm_out, size_t pcm_stride, int32_t* status_out,
                       void* cuda_stream);

/* One decode_frame (lc3_decoder.rs:217) for each listed stream; every other stream of the handle is untouched - the
 * reference's addressing by channel_index, for streams that have nothing to decode in a period (paused, not started,
 * finished, on another connection schedule: a lost frame would be concealed instead).
 *   stream_ids  HOST int32[n_rows]: row i of frames / frame_nbytes / pcm_out / status_out belongs to stream stream_ids[i].
 *               Any order; every id in [0, n_streams) and listed at most once, else LC3B_ERR_INVALID_ARG (the
 *               reference's bad channel_index panic, :228) and nothing is enqueued.  Only read during the call.
 *   n_rows      0 .. n_streams; 0 enqueues nothing and returns LC3B_OK.
 * Every other argument is what lc3b_decode_frames takes, with n_rows rows in place of n_streams.  A stream's PCM, status
 * and state are bit-identical to decoding its own frame sequence in a handle of its own, whatever mix of subset calls,
 * full calls, time-parallel calls and resets it went through.  The call follows the graph mode, lc3b_decoder_set_split,
 * set_dequant_mode (chosen by n_rows), set_synth_mode, set_min_nbytes and the stage mask, like lc3b_decode_frames; the
 * trace (lc3b_decoder_set_trace) is written per call row, like `frames`.  The ids are copied into the workspace (4 bytes
 * per stream, already counted by lc3b_decoder_workspace_bytes) with one cudaMemcpyAsync on `cuda_stream`. */
int lc3b_decode_frames_subset(lc3b_decoder* h, int bits_per_sample, const int32_t* stream_ids, int n_rows,
                              const uint8_t* frames, const int32_t* frame_nbytes, int nbytes, size_t frame_stride,
                              int16_t* pcm_out, size_t pcm_stride, int32_t* status_out, void* cuda_stream);
/* The listed streams get exactly the state lc3b_decoder_init gives a stream (a slot handed to a new call); no other
 * stream is touched.  stream_ids / n as in lc3b_decode_frames_subset. */
int lc3b_decoder_reset_streams(lc3b_decoder* h, const int32_t* stream_ids, int n, void* cuda_stream);

/* Same call with HOST buffers (what a caller of the reference holds): copies frames host->device, decodes, copies
 * PCM device->host, all on `cuda_stream`, using staging areas inside the workspace.  Asynchronous when the host
 * buffers are pinned.  status_out (host, nullable) as above. */
int lc3b_decode_frames_host(lc3b_decoder* h, int bits_per_sample, const uint8_t* frames, const int32_t* frame_nbytes,
                            int nbytes, size_t frame_stride, int16_t* pcm_out, size_t pcm_stride, int32_t* status_out,
                            void* cuda_stream);

/* Optional pipelining of lc3b_decode_frames_host.  Off (default): every copy and kernel rides `cuda_stream`, PCM is
 * valid once that stream has drained.  On: the device->host PCM copy of call i runs on an internal stream from a
 * double-buffered staging area and overlaps the kernels of call i+1; PCM of a call is valid after
 * lc3b_decoder_host_fence(h, s) followed by draining stream s (the fence makes s wait for all outstanding copies). */
int lc3b_decoder_set_host_pipelining(lc3b_decoder* h, int on);
int lc3b_decoder_host_fence(lc3b_decoder* h, void* cuda_stream);

/* Time-parallel decode (SURVEY.md 8f-1): `n_frames` consecutive frames of EVERY stream in one call - the whole-file
 * workflow of examples/decode.rs:85-123 without one launch per frame period.  Equivalent to n_frames calls of
 * lc3b_decode_frames (same PCM, same per-stream state afterwards, so the two entry points can be mixed freely).
 *   frames        device; frame f of stream s at frames + (s*n_frames + f)*frame_stride
 *   frame_nbytes  device int32[n_streams*n_frames] or NULL (as in lc3b_decode_frames; 0 = lost frame)
 *   pcm_out       device int16 [n_streams][n_frames*nf]: every stream's audio is contiguous in time
 *   status_out    device int32[n_streams*n_frames] or NULL
 *   scratch       device, at least lc3b_decoder_multi_scratch_bytes(h, n_frames) bytes, 256-byte aligned; caller-owned,
 *                 only used during the call */
int lc3b_decoder_multi_scratch_bytes(const lc3b_decoder* h, int n_frames, size_t* device_bytes);
int lc3b_decode_stream_frames(lc3b_decoder* h, int bits_per_sample, const uint8_t* frames, const int32_t* frame_nbytes,
                              int nbytes, size_t frame_stride, int n_frames, int16_t* pcm_out, int32_t* status_out,
                              void* scratch, size_t scratch_bytes, void* cuda_stream);

/* Time-parallel decode of a chosen subset of streams, each with its own number of frames: a batch of files of different
 * lengths in one handle, or per-stream jitter buffers of different depths, in one call.  Row i of the call advances
 * stream stream_ids[i] by frame_counts[i] frames and equals that many lc3b_decode_frames calls on it (same PCM, status
 * and per-stream state afterwards); streams not listed, and rows with count 0, are untouched.
 *   stream_ids, frame_counts  HOST int32[n_rows], only read during the call.  Ids as in lc3b_decode_frames_subset (any
 *               order, each in [0, n_streams) and at most once); counts >= 0.
 *   units       let off_i be the sum of frame_counts[0 .. i-1] (the caller's row order): frame f of row i is unit off_i + f,
 *               so each row's frames and audio are contiguous and rows follow each other in the caller's order
 *   frames      device; unit v at frames + v*frame_stride
 *   frame_nbytes, status_out  device int32[total] or NULL, one per unit (as in lc3b_decode_stream_frames)
 *   pcm_out     device int16; unit v at pcm_out + v*nf
 *   scratch     device, at least lc3b_decoder_multi_subset_scratch_bytes(h, n_rows, total) bytes, 256-byte aligned;
 *               caller-owned, only used during the call
 * total = sum of the counts.  Returns LC3B_OK and enqueues nothing when n_rows or total is 0; LC3B_ERR_INVALID_ARG for a
 * bad or duplicate id, a negative count, a total beyond 0x7fffffff / 512 and the argument errors of
 * lc3b_decode_stream_frames; LC3B_ERR_WORKSPACE for scratch that is too small or misaligned; LC3B_ERR_BITS_PER_SAMPLE
 * when bits_per_sample != 16.  Nothing is enqueued on an error.  The row table is copied to the front of the scratch with
 * one cudaMemcpyAsync on `cuda_stream`.  lc3b_decoder_set_split and set_dequant_mode apply as to
 * lc3b_decode_stream_frames, by the total. */
int lc3b_decoder_multi_subset_scratch_bytes(const lc3b_decoder* h, int n_rows, long long total_frames, size_t* device_bytes);
int lc3b_decode_stream_frames_subset(lc3b_decoder* h, int bits_per_sample, const int32_t* stream_ids, const int32_t* frame_counts,
                                     int n_rows, const uint8_t* frames, const int32_t* frame_nbytes, int nbytes,
                                     size_t frame_stride, int16_t* pcm_out, int32_t* status_out, void* scratch,
                                     size_t scratch_bytes, void* cuda_stream);

/* Inspection (parity gate i, SURVEY.md 8d): when set, every decode also writes, per stream, a record of
 * LC3B_TRACE_WORDS int32 (layout below) and the entropy-decoded integer spectrum x[0..ne).  Device pointers,
 * NULL to disable.  trace: [n_streams][LC3B_TRACE_WORDS], x: [n_streams][ne].  lc3b_decode_frames_subset writes
 * rows 0 .. n_rows-1, one per call row. */
int lc3b_decoder_set_trace(lc3b_decoder* h, int32_t* trace, int32_t* x);

/* Spectrum handed to the IMDCT by the last decode (after SNS, or the concealed one): device f32 [n_streams][ne],
 * copied into `out` (device) on `cuda_stream`.  For stage-level parity tests. */
int lc3b_decoder_get_spectrum(lc3b_decoder* h, float* out, void* cuda_stream);

/* How a call's kernels are issued: 0 = one launch per kernel on `cuda_stream`; 1 = the whole call as ONE CUDA graph
 * launch (graphs are cached per handle and keyed by the call's arguments; a caller cycling through a few buffer sets
 * replays instantiated graphs, anything else patches an executable graph in place).  Default: 1 for handles of at most
 * 131 072 streams (launch-sensitive), else 0; LC3B_GRAPH=0/1 in the environment overrides the default.  Results are
 * identical either way.  graph_stats: cache hits / in-place updates / instantiations so far (any pointer may be NULL). */
int lc3b_decoder_set_graph_mode(lc3b_decoder* h, int mode);
/* Into how many independent sub-batches of streams a call is cut: 0 = by batch size (the default: 4 from 65 536 streams,
 * 1 below), 1 = never, 2 or 4 = always.  The sub-batches' kernels run on auxiliary streams of the handle, forked from
 * and joined back into `cuda_stream` inside the call (or as parallel branches of the call's graph), so that one
 * sub-batch's kernels fill the SMs another's last wave leaves idle.  Streams are independent, so results are identical
 * for every setting.  LC3B_SPLIT=k in the environment overrides the default. */
int lc3b_decoder_set_split(lc3b_decoder* h, int k);
/* A promise about the frames this handle will see: every submitted frame is at least `min_nbytes` long or is a lost
 * frame (length 0).  Default 0 (no promise).  When the promised length rules the long-term post filter out for every
 * frame the handle accepts - the reference's gain table ends in the row (0.0, 0) once the frame carries 560 + 80 * fs_ind
 * bits per 10 ms (src/decoder/long_term_post_filter.rs:142-161), e.g. 110 bytes at 48 kHz / 10 ms - the decoder stops
 * keeping the filter's 20 / 22.5 ms output history (it can never be read again), which removes a quarter of the
 * synthesis kernel's memory traffic, and does not launch the post-filter kernel.  Results are bit-identical for every frame that
 * keeps the promise; a non-empty frame shorter than min_nbytes is treated as a lost frame (concealed), and a call whose
 * fixed `nbytes` is below it returns LC3B_ERR_INVALID_ARG.  Set it before the first decode. */
int lc3b_decoder_set_min_nbytes(lc3b_decoder* h, int min_nbytes);
/* Which synthesis (IMDCT + overlap-add) kernel runs: 0 = by launch size (default: two frames per warp for large
 * 48 / 44.1 kHz 10 ms launches, one frame per warp otherwise); 1 = always one frame per warp.  Bit-identical results;
 * the choice only matters for speed. */
int lc3b_decoder_set_synth_mode(lc3b_decoder* h, int mode);
/* Which dequantisation kernel runs: 0 = by batch size (default: one warp per frame up to 12 288 streams, one thread per
 * frame above), 1 = warp per frame, 2 = thread per frame.  Bit-identical results; the choice only matters for speed. */
int lc3b_decoder_set_dequant_mode(lc3b_decoder* h, int mode);
int lc3b_decoder_graph_stats(const lc3b_decoder* h, uint64_t* hits, uint64_t* updates, uint64_t* builds);

/* Profiling hook: which kernels lc3b_decode_frames launches (bit 0 = entropy kernel, bit 1 = dequantisation kernel,
 * bit 2 = synthesis kernel and the post-filter kernel behind it; default 7).  Lets bench.py time each kernel alone
 * with CUDA events; results are only meaningful with mask 7. */
int lc3b_decoder_set_stage_mask(lc3b_decoder* h, int mask);

void lc3b_decoder_destroy(lc3b_decoder* h);

/* ------------------------------------------------------------------ mixed-rate decoder (BASELINE config 4)
 * Lc3Decoder::new takes ONE frame duration and ONE sampling frequency for all its channels
 * (src/decoder/lc3_decoder.rs:181), so a mixed population of streams is a set of reference decoders.  This handle is
 * that set - up to twelve (sampling frequency, frame duration) configurations - driven as one batch: one entropy
 * launch over every stream, one dequantisation launch per frame duration, one synthesis + post-filter launch per
 * configuration, the whole call issued as one CUDA graph.
 *
 * Row order: streams are bucketed by configuration, buckets sorted by (sampling_frequency, frame_duration), streams of a
 * bucket in their original order.  lc3b_mixed_decoder_layout returns that order (`order[row]` = original stream id;
 * nullable) and the bucket table; the caller lays the rows of `frames`, `frame_nbytes`, `pcm_out`, `status_out` out in
 * that order, so every bucket is a contiguous row range and nothing is gathered or scattered on the device. */
typedef struct lc3b_mixed_decoder lc3b_mixed_decoder;
typedef struct lc3b_mixed_bucket {
    int32_t sampling_frequency, frame_duration;   /* LC3B_HZ*, LC3B_7P5MS / LC3B_10MS */
    int32_t first_row, n_rows;                    /* rows [first_row, first_row + n_rows) of the caller's buffers */
    int32_t nf, reserved;                         /* samples per frame of this bucket */
    uint64_t host_pcm_offset;                     /* lc3b_mixed_decode_frames_host: int16 offset of the bucket's dense PCM */
} lc3b_mixed_bucket;
#define LC3B_MIXED_MAX_BUCKETS 12
int lc3b_mixed_decoder_layout(int n_streams, const int32_t* sampling_frequency, const int32_t* frame_duration, int32_t* order,
                              lc3b_mixed_bucket* buckets /* [LC3B_MIXED_MAX_BUCKETS] */, int32_t* n_buckets,
                              uint64_t* host_pcm_elems);
/* Lc3Decoder::calc_working_buffer_lengths / Lc3Decoder::new for the whole set (sampling_frequency[s], frame_duration[s]
 * describe ORIGINAL stream s; host arrays, only read during the call). */
int lc3b_mixed_decoder_workspace_bytes(int n_streams, const int32_t* sampling_frequency, const int32_t* frame_duration,
                                       int max_nbytes, size_t* device_bytes);
int lc3b_mixed_decoder_init(lc3b_mixed_decoder** out, int n_streams, const int32_t* sampling_frequency,
                            const int32_t* frame_duration, int max_nbytes, int device, void* dev_workspace,
                            size_t workspace_bytes, void* cuda_stream);
/* One Lc3Decoder::decode_frame per stream (rows in bucket order, see above).  frame_nbytes is required (device
 * int32[n_streams]: configurations differ in frame length; 0 = lost frame); `nbytes` bounds it (<= max_nbytes, <= frame_stride).
 * pcm_out rows have one common pitch `pcm_stride` >= the largest nf; a row of bucket b receives nf_b samples. */
int lc3b_mixed_decode_frames(lc3b_mixed_decoder* h, int bits_per_sample, const uint8_t* frames, const int32_t* frame_nbytes,
                             int nbytes, size_t frame_stride, int16_t* pcm_out, size_t pcm_stride, int32_t* status_out,
                             void* cuda_stream);
/* Same with HOST buffers.  pcm_out is DENSE per bucket: bucket b's rows are [n_rows][nf_b] int16 at element offset
 * host_pcm_offset (lc3b_mixed_decoder_layout), host_pcm_elems in total - so the read-back is one linear copy. */
int lc3b_mixed_decode_frames_host(lc3b_mixed_decoder* h, int bits_per_sample, const uint8_t* frames, const int32_t* frame_nbytes,
                                  int nbytes, size_t frame_stride, int16_t* pcm_out, int32_t* status_out, void* cuda_stream);
int lc3b_mixed_decoder_set_host_pipelining(lc3b_mixed_decoder* h, int on);   /* as lc3b_decoder_set_host_pipelining */
int lc3b_mixed_decoder_host_fence(lc3b_mixed_decoder* h, void* cuda_stream);
int lc3b_mixed_decoder_set_graph_mode(lc3b_mixed_decoder* h, int mode);      /* default 1 (graph) */
int lc3b_mixed_decoder_set_dequant_mode(lc3b_mixed_decoder* h, int mode);    /* as lc3b_decoder_set_dequant_mode */
void lc3b_mixed_decoder_destroy(lc3b_mixed_decoder* h);

/* ------------------------------------------------------------------ encoder */
typedef struct lc3b_encoder lc3b_encoder;

/* Lc3Encoder::calc_working_buffer_lengths, src/encoder/lc3_encoder.rs:194.  8 kHz returns LC3B_ERR_INVALID_ARG:
 * Lc3Encoder::new panics there (BandwidthDetector::new indexes a table with fs_ind - 1, bandwidth_detector.rs:42-56). */
int lc3b_encoder_workspace_bytes(int n_streams, int frame_duration, int sampling_frequency, int max_nbytes,
                                 size_t* device_bytes);

/* Lc3Encoder::new, src/encoder/lc3_encoder.rs:117: zeroed working memory, t_prev = 17 (long_term_post_filter.rs:85),
 * attack_pos_last = -1 (attack_detector.rs:38). */
int lc3b_encoder_init(lc3b_encoder** out, int n_streams, int frame_duration, int sampling_frequency, int max_nbytes,
                      int device, void* dev_workspace, size_t workspace_bytes, void* cuda_stream);

/* One Lc3Encoder::encode_frame (src/encoder/lc3_encoder.rs:175) per stream.
 *   pcm_in      device int16, stream s at pcm_in + s*pcm_stride (elements), nf samples each (`samples_in`)
 *   frames_out  device, stream s at frames_out + s*frame_stride, `nbytes` bytes each (`buf_out`, buf_out.len() = nbytes)
 * The reference's encode cannot fail (Lc3EncoderError is empty, :30); wrong slice lengths panic there and are
 * LC3B_ERR_INVALID_ARG here (nbytes < 20 underflows the bit budget, spectral_quantization.rs:133). */
int lc3b_encode_frames(lc3b_encoder* h, const int16_t* pcm_in, size_t pcm_stride, uint8_t* frames_out, int nbytes,
                       size_t frame_stride, void* cuda_stream);
/* One encode_frame (lc3_encoder.rs:175) for each listed stream; every other stream of the handle is untouched.
 *   stream_ids  HOST int32[n_rows], as in lc3b_decode_frames_subset: row i of pcm_in / frames_out belongs to stream
 *               stream_ids[i]; ids in [0, n_streams), none twice, else LC3B_ERR_INVALID_ARG and nothing is enqueued.
 *   n_rows      0 .. n_streams; 0 enqueues nothing and returns LC3B_OK.
 * Every other argument is what lc3b_encode_frames takes, with n_rows rows.  A stream's bytes and state are identical to
 * encoding its own sequence in a handle of its own.  Follows the graph mode and the stage mask; lc3b_encoder_debug_read
 * then reports per call row.  The ids are copied into the workspace (4 bytes per stream, already counted by
 * lc3b_encoder_workspace_bytes) with one cudaMemcpyAsync on `cuda_stream`. */
int lc3b_encode_frames_subset(lc3b_encoder* h, const int32_t* stream_ids, int n_rows, const int16_t* pcm_in,
                              size_t pcm_stride, uint8_t* frames_out, int nbytes, size_t frame_stride, void* cuda_stream);
/* The listed streams get exactly the state lc3b_encoder_init gives a stream; no other stream is touched. */
int lc3b_encoder_reset_streams(lc3b_encoder* h, const int32_t* stream_ids, int n, void* cuda_stream);
/* Same with HOST buffers (pinned => asynchronous). */
int lc3b_encode_frames_host(lc3b_encoder* h, const int16_t* pcm_in, size_t pcm_stride, uint8_t* frames_out, int nbytes,
                            size_t frame_stride, void* cuda_stream);
/* Optional pipelining of lc3b_encode_frames_host.  Off (default): copies and kernels ride `cuda_stream`.  On: the
 * host->device PCM copy runs on an internal stream into a double-buffered staging area, so the upload of call i+1
 * overlaps the kernels of call i.  Results are ordered on `cuda_stream` as before (the bitstream copy stays on it);
 * the caller's PCM buffer must stay valid until the call's work has drained, as with any asynchronous copy. */
int lc3b_encoder_set_host_pipelining(lc3b_encoder* h, int on);
/* Time-parallel encode: `n_frames` consecutive frames of EVERY stream in one call - the whole-file workflow of
 * examples/encode.rs:73-116 without one launch per frame period.  Equivalent to n_frames calls of lc3b_encode_frames
 * with the same `nbytes` (same bytes, same per-stream state afterwards, so the two entry points can be mixed freely).
 *   pcm_in      device int16 [n_streams][n_frames*nf]: every stream's audio is contiguous in time
 *   frames_out  device; frame f of stream s at frames_out + (s*n_frames + f)*frame_stride, `nbytes` bytes each
 *   scratch     device, at least lc3b_encoder_multi_scratch_bytes(h, n_frames) bytes, 256-byte aligned; caller-owned,
 *               only used during the call
 * Returns LC3B_ERR_INVALID_ARG as lc3b_encode_frames does, and for n_frames < 1 or n_streams*n_frames beyond an int;
 * LC3B_ERR_WORKSPACE for scratch that is too small or misaligned.  The call follows lc3b_encoder_set_graph_mode (the
 * whole call is one graph launch in graph mode); the stage mask does not apply to it, and lc3b_encoder_debug_read keeps
 * reporting the last lc3b_encode_frames call (this call does not touch those buffers). */
int lc3b_encoder_multi_scratch_bytes(const lc3b_encoder* h, int n_frames, size_t* device_bytes);
int lc3b_encode_stream_frames(lc3b_encoder* h, const int16_t* pcm_in, int n_frames, uint8_t* frames_out, int nbytes,
                              size_t frame_stride, void* scratch, size_t scratch_bytes, void* cuda_stream);
/* Time-parallel encode of a chosen subset of streams, each with its own number of frames (the encoder twin of
 * lc3b_decode_stream_frames_subset, same ids, counts and unit layout).  Row i equals frame_counts[i] calls of
 * lc3b_encode_frames on stream stream_ids[i] with the same `nbytes` (same bytes and per-stream state afterwards); streams
 * not listed, and rows with count 0, are untouched.
 *   pcm_in      device int16; unit v at pcm_in + v*nf
 *   frames_out  device; unit v at frames_out + v*frame_stride, `nbytes` bytes each
 *   scratch     device, at least lc3b_encoder_multi_subset_scratch_bytes(h, n_rows, total) bytes, 256-byte aligned
 * Returns LC3B_OK and enqueues nothing when n_rows or total is 0; LC3B_ERR_INVALID_ARG for a bad or duplicate id, a
 * negative count, a total beyond INT32_MAX and the argument errors of lc3b_encode_stream_frames; LC3B_ERR_WORKSPACE for
 * scratch that is too small or misaligned.  Nothing is enqueued on an error.  Follows lc3b_encoder_set_graph_mode like
 * lc3b_encode_stream_frames; the row table goes to the front of the scratch with one cudaMemcpyAsync on `cuda_stream`. */
int lc3b_encoder_multi_subset_scratch_bytes(const lc3b_encoder* h, int n_rows, long long total_frames, size_t* device_bytes);
int lc3b_encode_stream_frames_subset(lc3b_encoder* h, const int32_t* stream_ids, const int32_t* frame_counts, int n_rows,
                                     const int16_t* pcm_in, uint8_t* frames_out, int nbytes, size_t frame_stride, void* scratch,
                                     size_t scratch_bytes, void* cuda_stream);
int lc3b_encoder_set_graph_mode(lc3b_encoder* h, int mode);   /* as lc3b_decoder_set_graph_mode */
/* Test hook: device copies of the last encode's intermediates (any pointer may be NULL): xf [S][ne] f32 (quantiser
 * input, after SNS and TNS), e_b [S][64] f32, hand [S][8] i32 (near_nyquist, attack, pitch_index, pitch_present,
 * ltpf_active, nbits_ltpf), xq [S][ne] i16.  After lc3b_encode_frames_subset, row i is call row i (rows from n_rows on
 * are left from earlier calls). */
int lc3b_encoder_debug_read(lc3b_encoder* h, float* xf, float* e_b, int32_t* hand, int16_t* xq, void* cuda_stream);
/* Profiling hook, like lc3b_decoder_set_stage_mask: bit 0 = MDCT kernel, bit 1 = attack/LTPF analysis kernel,
 * bit 2 = SNS kernel (with the bandwidth detector), bit 3 = TNS kernel, bit 4 = quantise kernel, bit 5 = the
 * bitstream stage (prepare, range coder, finish kernels).  Default 63 (all). */
int lc3b_encoder_set_stage_mask(lc3b_encoder* h, int mask);
void lc3b_encoder_destroy(lc3b_encoder* h);

/* ------------------------------------------------------------------ one batch over the GPUs of a box (SURVEY.md 8e)
 * Streams never interact (DecoderChannel / EncoderChannel own all state, src/decoder/lc3_decoder.rs:62-69,
 * src/encoder/lc3_encoder.rs:42-60), so a batch shards by stream id with nothing to exchange: stream s belongs to
 * shard floor(s * G / N) - a contiguous block of rows per GPU; no collective, no peer access.
 * A sharded handle owns per GPU: a decoder / encoder handle on its own device workspace (allocated once, at create;
 * nothing afterwards), a CUDA stream and one host thread that issues that GPU's copies and launches.  The calls take
 * HOST buffers of the whole batch (pin them: lc3b_host_alloc, or cudaHostAlloc with the portable flag), hand every
 * thread its row range and return at once; *_wait joins all outstanding calls, after which the outputs are valid and the
 * first error of any shard is returned.  Calls must come from one thread at a time; frames of a stream stay in order.
 *   devices   n_devices CUDA device indices, or NULL for 0 .. n_devices-1
 *   *_shard   which device and rows [first_stream, first_stream + n_streams) a shard covers */
typedef struct lc3b_sharded_decoder lc3b_sharded_decoder;
int lc3b_sharded_decoder_create(lc3b_sharded_decoder** out, int n_streams, int frame_duration, int sampling_frequency,
                                int max_nbytes, const int* devices, int n_devices);
int lc3b_sharded_decoder_n_shards(const lc3b_sharded_decoder* h);
int lc3b_sharded_decoder_shard(const lc3b_sharded_decoder* h, int shard, int* device, int* first_stream, int* n_streams);
/* arguments as lc3b_decode_frames_host, for all n_streams rows */
int lc3b_sharded_decode_frames_host(lc3b_sharded_decoder* h, int bits_per_sample, const uint8_t* frames,
                                    const int32_t* frame_nbytes, int nbytes, size_t frame_stride, int16_t* pcm_out,
                                    size_t pcm_stride, int32_t* status_out);
int lc3b_sharded_decoder_wait(lc3b_sharded_decoder* h);
int lc3b_sharded_decoder_set_min_nbytes(lc3b_sharded_decoder* h, int min_nbytes);   /* lc3b_decoder_set_min_nbytes on every shard */
void lc3b_sharded_decoder_destroy(lc3b_sharded_decoder* h);

typedef struct lc3b_sharded_encoder lc3b_sharded_encoder;
int lc3b_sharded_encoder_create(lc3b_sharded_encoder** out, int n_streams, int frame_duration, int sampling_frequency,
                                int max_nbytes, const int* devices, int n_devices);
int lc3b_sharded_encoder_n_shards(const lc3b_sharded_encoder* h);
int lc3b_sharded_encoder_shard(const lc3b_sharded_encoder* h, int shard, int* device, int* first_stream, int* n_streams);
/* arguments as lc3b_encode_frames_host, for all n_streams rows */
int lc3b_sharded_encode_frames_host(lc3b_sharded_encoder* h, const int16_t* pcm_in, size_t pcm_stride, uint8_t* frames_out,
                                    int nbytes, size_t frame_stride);
int lc3b_sharded_encoder_wait(lc3b_sharded_encoder* h);
void lc3b_sharded_encoder_destroy(lc3b_sharded_encoder* h);

/* Pinned (page-locked, portable across devices) host memory for the host-buffer entry points, for callers that do
 * not link the CUDA runtime themselves. */
int lc3b_host_alloc(void** out, size_t bytes);
void lc3b_host_free(void* p);

/* Self-test hooks: the engine's own f32 transcendentals (csrc/lc3b_math.cuh, msun-style, see DESIGN.md) evaluated
 * on the host (no GPU needed) or on the device, so tests can compare them with the oracle's.
 * which: 0 powf(x,y) 1 log2f 2 log10f 3 exp2f 4 asinf 5 exp2_raw(fast-math) 6 powi(x,(int)y).
 * Host variant: x, y, out are host arrays.  Device variant: device arrays, runs on cuda_stream. */
int lc3b_selftest_math_host(int which, const float* x, const float* y, float* out, int n);
int lc3b_selftest_math_device(int which, const float* x, const float* y, float* out, int n, void* cuda_stream);

/* trace record layout (int32 words) */
enum {
    LC3B_TR_OK = 0, LC3B_TR_BW, LC3B_TR_LASTNZ, LC3B_TR_LSB_MODE, LC3B_TR_GG_IND, LC3B_TR_NUM_TNS,
    LC3B_TR_RC_ORDER_IN0, LC3B_TR_RC_ORDER_IN1, LC3B_TR_IND_LF, LC3B_TR_IND_HF, LC3B_TR_LS_INDA, LC3B_TR_LS_INDB,
    LC3B_TR_IDX_A, LC3B_TR_IDX_B, LC3B_TR_SUBMODE_LSB, LC3B_TR_SUBMODE_MSB, LC3B_TR_G_IND, LC3B_TR_PITCH_PRESENT,
    LC3B_TR_LTPF_ACTIVE, LC3B_TR_PITCH_INDEX, LC3B_TR_NOISE_FACTOR, LC3B_TR_RC_ORDER0, LC3B_TR_RC_ORDER1,
    LC3B_TR_RC_I0 /* 16 words */, LC3B_TR_NRES = LC3B_TR_RC_I0 + 16, LC3B_TR_SEED, LC3B_TR_IS_ZERO,
    LC3B_TRACE_WORDS = 48
};

#ifdef __cplusplus
}
#endif
#endif /* LC3B_H */
