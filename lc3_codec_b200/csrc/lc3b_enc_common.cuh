// lc3b engine: encoder declarations shared by the two encoder kernels and the C ABI.
//
// The encoder's bitstream must be byte-identical to the reference's, so every f32 operation that feeds a decision
// is performed in the reference's order WITHOUT fused multiply-add: the encoder translation units are compiled
// with -fmad=false (see Makefile), which lets the code below use ordinary a*b+c expressions.
#pragma once
#include "lc3b_common.cuh"

namespace lc3b {

// per-config constants of the encoder (device memory, built at init)
struct EncConfig {
    int32_t fs_ind, fs, ne, nb, nf, z, n_ms;
    int32_t n_fft;
    int32_t n_levels;                 // kissfft factor levels
    int32_t fac_p[8], fac_m[8], fac_stride[8];   // kf_factor (kissfft.rs:47): radix, sub-length, fstride per level
    int32_t band_idx[65];
    uint8_t band_of[400];             // line -> band (255: beyond the last band)
    float band_width_of[400];         // line -> width of its band as f32, 0 beyond the last band (energy estimation divides by it)
    // LTPF analysis (encoder/long_term_post_filter.rs:91-124)
    int32_t len12p8, len6p4, delay, up, x_s_ext_len, x12_len;
    float resamp_fac;
    float resamp_ph[240];             // TAB_RESAMP_FILTER in phase-major order: [r][j] = h[up (j - 120/up + 1) - r], 0 outside (-120, 120)
    // attack detector (attack_detector.rs:24-43)
    int32_t att_num_ds, att_num_blocks, att_pos_limit;
    float tns_sin[17];
    float gg_table[400];              // 10^((i - 245) / 28) via powf_msun (spectral_quantization.rs:239)
    float pre_emph[64];               // 10^(b * g_tilt / 630) via powf_msun (spectral_noise_shaping.rs:216-219)
};

// hand-off record analysis kernel -> quantisation kernel (int32 words per stream)
enum {
    EH_NEAR_NYQUIST = 0, EH_ATTACK, EH_PITCH_INDEX, EH_PITCH_PRESENT, EH_LTPF_ACTIVE, EH_NBITS_LTPF, EH_WORDS = 8
};
constexpr int QH_WORDS = 40;

// per-stream persistent scalars of the encoder (int32 words; floats as bits)
enum {
    ES_ATT_ENERGY_LAST = 0, ES_ATT_MAX_ENERGY_LAST, ES_ATT_POS_LAST, ES_ATT_TM1, ES_ATT_TM2,   // attack_detector.rs:17-21
    ES_H50_M1, ES_H50_M2, ES_T_PREV, ES_MEM_PITCH, ES_MEM_NC, ES_MEM_MEM_NC, ES_MEM_LTPF_ACTIVE,   // long_term_post_filter.rs:31-41
    ES_Q_RESET_OFFSET_OLD, ES_Q_NBITS_OFFSET_OLD, ES_Q_NBITS_EST_OLD,                          // spectral_quantization.rs:57-60
    ES_WORDS = 16
};

struct EncoderState {
    lc3b_config cfg;
    int n_streams, max_nbytes, device;
    EncConfig* ecfg;
    float* win;            // [2*nf]  w_N (unmodified)
    float2* dtw;           // [n_fft] DCT-IV twiddles
    float2* ftw;           // [n_fft] kissfft twiddles
    int32_t* perm;         // [n_fft] kissfft leaf permutation: work[o] = in[perm[o]]
    int16_t* thist;        // [S][nf - z]   last nf-z input samples (encoder/modified_dct.rs:126-138)
    int16_t* xs_hist;      // [S][64]       last 240/up input samples (long_term_post_filter.rs:217-224)
    float* x12;            // [S][x12_len]  x_tilde_12p8d_extended
    float* x6;             // [S][178]      x_6p4_extended
    int32_t* estate;       // [S][ES_WORDS]
    float* xf;             // [S][ne]       MDCT spectrum -> shaped -> TNS filtered (in place)
    float* e_b;            // [S][64]
    int32_t* ehand;        // [S][EH_WORDS]
    int16_t* xq;           // [S][ne]       quantised spectrum
    int32_t* qhand;        // [S][QH_WORDS] decisions handed from kernel to kernel (lc3b_enc_quant.cu)
    uint8_t* lsbs;         // [S][ne]       deferred LSBs / sign bits in lsb_mode (bitstream_encoding.rs:22)
    uint32_t* bs_scratch;  // [S][bs_words] bitstream hand-off: job record, tail bits, side bits, symbol queue, forward bytes
    int bs_words;          //               32-bit words per stream of bs_scratch (for max_nbytes)
    int16_t* stage_in;     // [S][nf]       staging for the host entry point
    uint8_t* stage_out;    // [S][max_nbytes]
    int32_t* ids;          // [S]           id list of the current subset call (lc3b_encode_frames_subset, lc3b_encoder_reset_streams)
};

cudaError_t prepare_enc_analysis(const EncoderState& st);   // shared-memory limits of the kernels, once per handle
cudaError_t prepare_enc_quant(const EncoderState& st);
int enc_bitstream_scratch_words(int ne, int max_nbytes);   // per-stream size of EncoderState::bs_scratch
// The encoder's launches, written into a plan (lc3b_plan.cuh).
// stages of plan_enc_analysis: bit 0 MDCT kernel, bit 1 attack detector + LTPF analysis kernel; of plan_enc_quant: bit 0
// SNS kernel (with the bandwidth detector), bit 1 TNS kernel, bit 2 quantise kernel, bit 3 bitstream kernels.
// ids: a subset call, `st` a view whose st.n_streams is the call's row count; row u's persistent state (thist, xs_hist,
// x12, x6, estate) is that of handle stream ids[u] (device memory), every other buffer has a row per call row.
// rows: a time-parallel call, `st` a view whose st.n_streams is the call's unit count and whose per-frame buffers have a
// row per unit; its per-stream state (xs_hist, x12, x6, estate) keeps a row per stream.  The attack / LTPF kernel and
// the quantise kernel run a warp per row of the device row table (n_rows rows with frames, lc3b_common.cuh), walking the
// row's units in order; every other kernel runs per unit.
struct LaunchPlan;
void plan_enc_analysis(LaunchPlan& plan, const EncoderState& st, const int16_t* pcm, size_t pcm_stride, int nbytes, int stages,
                       const int32_t* ids = nullptr, const int32_t* rows = nullptr, int n_rows = 0);
void plan_enc_quant(LaunchPlan& plan, const EncoderState& st, uint8_t* frames_out, int nbytes, size_t frame_stride, int stages,
                    const int32_t* ids = nullptr, const int32_t* rows = nullptr, int n_rows = 0);
// time-parallel encode (lc3b_enc_multi.cu) as one plan: n_rows listed rows, `total` units.  dense_frames > 0: a dense
// call, n_rows = n_live = the handle's streams of dense_frames frames each, whose row table the plan writes itself;
// otherwise the row table (n_live rows with frames) is at the front of the scratch (RowTable::send).
size_t enc_multi_scratch_bytes(const EncoderState& st, int n_rows, long long total);
void plan_enc_multi(LaunchPlan& plan, const EncoderState& st, const int16_t* pcm, int n_rows, int n_live, long long total,
                    int dense_frames, uint8_t* frames_out, int nbytes, size_t frame_stride, void* scratch);

}  // namespace lc3b
