// lc3b engine: shared declarations (host + device).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/lc3b.h"

#if defined(__CUDACC__)
#define LC3_TABLE(T) static __device__ const T
#else
#define LC3_TABLE(T) static const T
#endif

// Lane-strided loops with a warp-uniform trip count.  `for (i = lane; i < n; i += 32)` gives the lanes different trip
// counts; the warp then splits and was observed to stay split through the following uniform code (every later
// instruction issued twice, ncu thr/inst = 16).  Here every lane runs ceil(n/32) iterations with a predicated body.
#define WARP_STRIDE(v, n) for (int v##_b = 0, v = lane; v##_b < (n); v##_b += 32, v += 32) if (v < (n))
#define WARP_STRIDE_FROM(v, start, n) for (int v##_b = (start), v = (start) + lane; v##_b < (n); v##_b += 32, v += 32) if (v < (n))
// The same loops kept rolled, for the kernels that run through a lot of code once per frame and are bound by instruction
// fetch (ncu `no_instructions`: SNS and the bitstream stage): there code size matters more than the unrolled loads' overlap.
#define WARP_STRIDE_R(v, n) _Pragma("unroll 1") WARP_STRIDE(v, n)
#define WARP_STRIDE_FROM_R(v, start, n) _Pragma("unroll 1") WARP_STRIDE_FROM(v, start, n)

namespace lc3b {

constexpr int MAX_NE = 400;
constexpr int MAX_NF = 480;
constexpr int MAX_NBYTES = 400;      // LC3 frames are at most 400 bytes
constexpr int SIDE_WORDS = 16;       // dequantisation -> synthesis hand-off record, int32 words per stream
constexpr int HO_WORDS = 44;         // entropy -> dequantisation hand-off record, int32 words per thread slot

// hand-off record written by the entropy kernel for the synthesis kernel
enum {
    SD_OK = 0,          // 1: frame decoded; 0: conceal (lc3_decoder.rs:138-141)
    SD_LTPF_ACTIVE,     // LongTermPostFilterInfo.is_active
    SD_PITCH_INDEX,
    SD_NBITS,           // buf_in.len() * 8
    SD_PLC_SEED,        // PLC LCG state BEFORE this frame's ne steps (concealed frames)
    SD_PLC_ALPHA,       // f32 bits: alpha to apply (concealed frames)
    SD_SLOT,            // which of the two spectrum slots holds the spectrum to transform
    SD_SRC,             // time-parallel path: unit whose spectrum to transform (-2 own, -1 the handle's last good slot)
    SD_BLK,             // LTPF ring block of this frame's x_hat (synthesis kernel -> ltpf_kernel)
};
constexpr int XTAIL_FLOATS = 3 * 16;   // per stream: last 16 samples of x_hat of the frame in each ring block

// Subset calls (lc3b_decode_frames_subset, lc3b_encode_frames_subset) keep two indices apart: the ROW u of the call, which
// indexes its I/O and every per-call buffer, and the STATE ROW, the handle stream ids[u] whose persistent buffers the row
// reads and writes.  IDS is a template parameter of the kernels, so the dense instantiations (IDS = false) compile to
// exactly the code they had before the indirection existed.
template <bool IDS>
__device__ __forceinline__ int state_row(const int32_t* ids, int u) {
    if constexpr (IDS) return __ldg(ids + u);
    else return u;
}

// Time-parallel calls (lc3b_decode_stream_frames, lc3b_encode_stream_frames and their _subset forms) list their rows in a
// device ROW TABLE of RT_WORDS int32 per row: the state row (handle stream) the row advances, its first unit and its frame
// count.  A row's units are consecutive; the table holds only rows with frames, sorted by count, descending (RowTable in
// lc3b_handles.cuh), so the rows of a CTA that still have frame f are always the CTA's first rows.  A dense call's table
// is the identity {r, r * F, F}, which unit_rows_kernel writes on the device (already in that order).
constexpr int RT_WORDS = 3;
enum { RT_ROW = 0, RT_OFF, RT_COUNT };
struct RowSpan { int row, off, count; };
__device__ __forceinline__ RowSpan row_span(const int32_t* rows, int r) {
    return RowSpan{__ldg(rows + RT_WORDS * r + RT_ROW), __ldg(rows + RT_WORDS * r + RT_OFF), __ldg(rows + RT_WORDS * r + RT_COUNT)};
}
// unit_row[v] of a time-parallel call (plan_unit_rows): the state row of unit v's row, bit-inverted for the row's first unit
__device__ __forceinline__ int unit_state_row(int u) { return u < 0 ? ~u : u; }

// Everything a kernel needs to know about the (fs, duration) configuration; lives in the workspace.
struct DevConfig {
    int32_t fs_ind, fs, ne, nb, nf, z, n_ms;
    int32_t nbits_bw, lastnz_bits;       // side-info field widths
    int32_t n_fft;                       // nf / 2
    int32_t fft_radix[8];                // Stockham stage radices, product = n_fft, 0-terminated
    int32_t ltpf_l_den, ltpf_l_num, ltpf_blocks, ltpf_norm, ltpf_s2p5;
    int32_t band_idx[65];                // I_fs
    float gg_table[400];                 // 10^(i/28), i = index - 245  (global_gain.rs:19-20)
    float tns_sin[17];                   // sin(pi/17 * (i - 8)) (temporal_noise_shaping.rs:44)
    float ltpf_num[4][12];               // 0.85 * gain * TAB_LTPF_NUM[gain_ind][k]  (long_term_post_filter.rs:232-236)
    float ltpf_den[4][4][16];            // gain * TAB_LTPF_DEN[pitch_frac][k], first index = gain_ind
    uint32_t nf_lcg[MAX_NE + 1];         // noise-filling LCG jumped n steps: s_n = ((v >> 16) * s_0 + (v & 0xffff)) & 0xffff (noise_filling.rs:49)
    // per-config float tables appended after this struct in the workspace:
    //   win  [2*nf]   gain * w[2nf-1-m]   (modified_dct.rs:89 and :131-134 folded together)
    //   dtw  [n_fft]  DCT-IV twiddles exp(-i*pi*(8n+1)/(8*nf)) as float2 (dct_iv.rs:30-35)
    //   ftw  [n_fft]  FFT twiddles exp(-2*pi*i*k/n_fft) as float2 (kissfft.rs:19-29)
};

struct DecoderState {
    // configuration
    lc3b_config cfg;
    int n_streams, n_blocks32, max_nbytes, device;
    int fixed_slot;      // -1: double-buffered spectrum slots tracked in sstate; >= 0: always write that slot (time-parallel path)
    int no_ltpf;         // 1: every frame the handle accepts is too long for the post filter to be active (gain row (0.0, 0))
    int min_nbytes;      // promised minimum frame length (0 = none), lc3b_decoder_set_min_nbytes
    int sm_count;        // multiprocessors of the handle's device (the launch size from which synthesis takes two frames per warp)
    int synth_mode;      // 0 synthesis kernel by launch size (default), 1 one frame per warp always (lc3b_decoder_set_synth_mode)
    int dequant_mode;    // 0 auto, 1 warp-per-frame dequantisation kernel, 2 thread-per-frame (lc3b_decoder_set_dequant_mode)
    // device pointers (carved from the caller's workspace)
    DevConfig* dcfg;
    float* win;          // [2*nf]
    float2* dtw;         // [n_fft]
    float2* ftw;         // [n_fft]
    uint8_t* sym_lut;    // [64][32] arithmetic-decoder symbol at the start of each 32-quotient bucket, built at init
    float* spec;         // [2][n_streams][ne]  double-buffered spectrum; the valid slot doubles as PLC "last good"
    int32_t* xq;         // [n_blocks32][ne][32] entropy-decoded integers, lane-interleaved (entropy -> dequantisation kernel)
    int32_t* handoff;    // [n_blocks32 * 32][HO_WORDS] decoded side information etc. (entropy -> dequantisation kernel)
    float* gband;        // [thread slots][64] SNS band gains, dequant_warp_kernel -> tns_list_kernel
    int32_t* tns_list;   // [2 + thread slots] count, CTAs done, thread slots of the frames tns_list_kernel has to finish (zero between calls)
    int32_t* nsym_prev;  // [n_streams] symbols decoded in the stream's previous good frame: predicts this frame's work (entropy kernel's sort key)
    float* ola;          // [n_streams][nf - z]  mem_ola_add (modified_dct.rs:16)
    float* ltpf_y;       // [n_streams][blocks*nf]  x_hat_ltpf_mem (long_term_post_filter.rs:30)
    float* ltpf_xtail;   // [n_streams][3][16]  last samples of x_hat_mem per ring block (only l_num <= 10 are ever read back)
    float* ltpf_x;       // [n_streams][nf]  x_hat of the current frame while its stream is inside an LTPF-active span
    int32_t* side;       // [n_streams][SIDE_WORDS]
    int32_t* sstate;     // [n_streams][8]  per-stream scalars, see SS_* below
    uint8_t* stage_in;   // [n_streams][max_nbytes] staging for the host-buffer entry point
    int16_t* stage_out;  // [n_streams][nf]
    int32_t* stage_len;  // [n_streams]
    int32_t* stage_status;  // [n_streams]
    int32_t* ids;        // [n_streams] id list of the current subset call (lc3b_decode_frames_subset, lc3b_decoder_reset_streams)
    // optional inspection outputs (caller-owned device memory)
    int32_t* trace;
    int32_t* trace_x;
};

// per-stream persistent scalars
enum {
    SS_SLOT = 0,        // index of the spectrum slot that holds the last good spectrum
    SS_PLC_LOST,        // num_lost_frames (packet_loss_concealment.rs:11)
    SS_PLC_ALPHA,       // f32 bits
    SS_PLC_SEED,        // plc_seed
    SS_LTPF_PREV,       // bit0 = ltpf_active_prev, bits 8.. = previous gain code (0..3 table row, 4 = zero gain)
    SS_LTPF_PINT,       // p_int_mem
    SS_LTPF_PFR,        // p_fr_mem
    SS_LTPF_BLK,        // block_start_index / nf
    SS_WORDS = 8
};

// Parameters of the entropy / dequantisation kernels (one struct, passed by value)
struct EntropyParams {
    const DevConfig* cfg;
    const uint8_t* frames;
    const int32_t* frame_nbytes;
    int nbytes;
    size_t frame_stride;
    int n_streams;        // streams of THIS launch (a sub-batch of the handle's streams when a call is split)
    int slot_streams;     // streams per spectrum slot = the handle's stream count (stride between the two slots)
    float* spec;          // [2][slot_streams][ne], offset to the launch's first stream
    int32_t* xq;          // [n_blocks32][ne][32]
    int32_t* handoff;     // [n_blocks32 * 32][HO_WORDS] entropy kernel -> dequantisation kernel
    int32_t* side;        // [n_streams][SIDE_WORDS]
    int32_t* sstate;      // [n_streams][SS_WORDS]
    int32_t* status_out;  // nullable
    int32_t* trace;       // nullable
    int32_t* trace_x;     // nullable
    const uint8_t* sym_lut;   // [64][32] symbol at the start of each 32-quotient bucket (init_sym_lut_kernel)
    float* gband;         // [thread slots][64] SNS band gains of frames waiting for the lattice kernel
    int32_t* tns_list;    // [2 + thread slots]: count, CTAs done, then the thread slots of frames with an active TNS filter
    int32_t* nsym_prev;   // [n_streams] arithmetic symbols the stream's previous good frame took (work-sorting key), nullable
    int fixed_slot;           // >= 0: spectrum always goes to this slot and sstate is left alone (time-parallel path)
    int min_nbytes;           // frames shorter than this (but not empty) break the handle's promise and are treated as lost
    int row_pitch;        // bytes per staged frame row in shared memory
    const int32_t* ids;   // subset call: row u of this launch is handle stream ids[u] (the IDS instantiations only)
};

// Mixed-rate batches: one (fs, duration) bucket = a contiguous row range of the caller's buffers with its own state.
// `ep` carries the bucket's static pointers; the per-call ones are patched in by the kernel (mixed_select).
struct MixedBucket {
    EntropyParams ep;
    int first_row;        // first row of the bucket in the caller's (bucket-ordered) buffers
    int first_cta;        // first CTA of the bucket in this table's launch
};
struct MixedParams {
    const MixedBucket* buckets;   // device
    int n_buckets;
    const uint8_t* frames;
    const int32_t* frame_nbytes;
    int nbytes;
    size_t frame_stride;
    int32_t* status_out;
    int row_pitch;
};
struct MixedTables {              // device tables + launch sizes: every bucket, the 10 ms ones, the 7.5 ms ones
    const MixedBucket *all, *b10, *b75;
    int n_all, n_10, n_75;
    int cta_all, cta_10, cta_75;
    int n_streams, dequant_mode;
};

struct LaunchPlan;
int entropy_row_pitch(int nbytes);
bool use_dequant_warp(int n_streams, int mode);   // mode: 0 auto (by batch size), 1 warp-per-frame, 2 thread-per-frame
// base / count: the sub-batch of the handle's streams the launches cover (base a multiple of 128; count < 0 = all);
// first_dep: what the first node added waits for (-2 = the node added just before, -1 = nothing)
// ids: a subset call's device id list (nullptr = a dense call, row u is stream u).  With ids, base / count cut the call's
// rows and the state pointers stay at the handle's first stream; n_rows is the call's row count (the dequantisation
// kernel is chosen by it).
EntropyParams entropy_params(const DecoderState& st, const uint8_t* frames, const int32_t* frame_nbytes, int nbytes,
                             size_t frame_stride, int32_t* status_out, int base = 0, int count = -1,
                             const int32_t* ids = nullptr);
void plan_entropy(LaunchPlan& plan, const DecoderState& st, const uint8_t* frames, const int32_t* frame_nbytes, int nbytes,
                  size_t frame_stride, int32_t* status_out, int stages, int base = 0, int count = -1, int first_dep = -2,
                  const int32_t* ids = nullptr, int n_rows = 0);
void plan_entropy_mixed(LaunchPlan& plan, const MixedTables& t, const uint8_t* frames, const int32_t* frame_nbytes, int nbytes,
                        size_t frame_stride, int32_t* status_out, int* node_d10, int* node_d75);
int plan_synth(LaunchPlan& plan, const DecoderState& st, int16_t* pcm_out, size_t pcm_stride, int dep, int base = 0, int count = -1,
               const int32_t* ids = nullptr);

cudaError_t prepare_entropy(const DecoderState& st);   // shared-memory limits of the kernels, once per handle
cudaError_t prepare_synth(const DecoderState& st);
cudaError_t launch_init_state(const DecoderState& st, cudaStream_t stream);

// time-parallel decode (SURVEY.md 8f-1), lc3b_dec_multi.cu: n_rows listed rows, `total` units.  dense_frames > 0: a dense
// call, n_rows = n_live = the handle's streams of dense_frames frames each, whose row table the call writes itself;
// otherwise the row table (n_live rows with frames) is at the front of the scratch already (RowTable::send).
int decode_split_min_streams();    // from this many streams (or units) a decode call is cut into sub-batches
size_t multi_scratch_bytes(const DecoderState& st, int n_rows, long long total);
cudaError_t prepare_multi(const DecoderState& st);
cudaError_t launch_decode_multi(const DecoderState& st, const uint8_t* frames, const int32_t* frame_nbytes, int nbytes,
                                size_t frame_stride, int n_rows, int n_live, long long total, int dense_frames, int16_t* pcm_out,
                                int32_t* status_out, void* scratch, cudaStream_t stream, struct PlanLanes* lanes);
// one kernel writing unit_row[v] for the units of the n_live rows of a device row table (shared with the encoder); with
// dense_frames > 0 it first writes the identity table of n_live rows of dense_frames frames
void plan_unit_rows(struct LaunchPlan& plan, int32_t* rows, int n_live, int dense_frames, int32_t* unit_row);

}  // namespace lc3b
