// CPU ORACLE - TEST INFRASTRUCTURE, NOT PRODUCT.
//
// A C++17 restatement of ninjasource/lc3-codec (Rust, `/root/reference`, cannot be
// compiled in this environment: no cargo/rustc) used ONLY as the parity checker by
// tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
// legs.  Nothing under lc3_codec_b200/ includes, links or calls this code.
//
// Parity pinning: every golden vector the reference's own unit tests hold (39
// #[test] functions, extracted mechanically into tests/golden/ by
// tools/extract_golden.py) is replayed against this code with exact equality in
// tests/test_oracle_golden.py.  Anything the reference's tests do not cover
// (7.5 ms, rates other than 48 kHz, lsb_mode, PLC/LTPF inside a full decode,
// encoder frames >= 2) is pinned only by "follows the cited Rust lines".
//
// Rules of the restatement (SURVEY.md section 7 "hard parts"):
//  * f32 arithmetic in the reference's operation order, no FMA contraction
//    (build with -ffp-contract=off, no -ffast-math);
//  * Rust `as` casts saturate and map NaN to 0 (rust_cast_* below);
//  * integer sums wrap (release build); usize arithmetic is 64-bit;
//  * f32 transcendentals are the `libm` crate's (FreeBSD msun ports), restated in
//    lc3o_math.cpp, because num-traits is built with `features = ["libm"]`
//    (Cargo.toml:17) under #![no_std] (src/lib.rs:1);
//  * `fast_math::exp2_raw` (Cargo.toml:19, decoder/spectral_noise_shaping.rs:122)
//    is restated from its published algorithm (fast-math 0.1.1).
#pragma once
#include <cmath>
#include <cstdint>
#include <cstring>
#include <vector>

#define LC3_TABLE(T) static const T
#include "../lc3_codec_b200/csrc/lc3_tables.h"

namespace lc3o {

// ---------------------------------------------------------------- config
// common/config.rs:2-100
enum SamplingFrequency { Hz8000 = 0, Hz16000, Hz24000, Hz32000, Hz44100, Hz48000 };
enum FrameDuration { SevenPointFiveMs = 0, TenMs = 1 };

struct Config {
    int fs_ind, fs, ne, nb, nf, z;
    FrameDuration n_ms;
};
Config make_config(SamplingFrequency sf, FrameDuration fd);
const uint16_t* band_indices(const Config& c);   // I_fs table for (fs_ind, n_ms)
const float* mdct_window(const Config& c);       // w_N table, 2*nf entries

// ---------------------------------------------------------------- rust semantics
static inline int32_t rust_f32_to_i32(float x) {
    if (x != x) return 0;
    if (x >= 2147483648.0f) return INT32_MAX;
    if (x <= -2147483648.0f) return INT32_MIN;
    return (int32_t)x;
}
static inline int16_t rust_f32_to_i16(float x) {
    if (x != x) return 0;
    if (x >= 32767.0f) return INT16_MAX;
    if (x <= -32768.0f) return INT16_MIN;
    return (int16_t)x;
}
static inline int8_t rust_f32_to_i8(float x) {
    if (x != x) return 0;
    if (x >= 127.0f) return INT8_MAX;
    if (x <= -128.0f) return INT8_MIN;
    return (int8_t)x;
}
static inline uint16_t rust_f32_to_u16(float x) {
    if (x != x) return 0;
    if (x >= 65535.0f) return UINT16_MAX;
    if (x <= 0.0f) return 0;
    return (uint16_t)x;
}
static inline uint64_t rust_f32_to_usize(float x) {
    if (x != x || x <= 0.0f) return 0;
    if (x >= 18446744073709551616.0f) return UINT64_MAX;
    return (uint64_t)x;
}
static inline uint64_t rust_f64_to_usize(double x) {
    if (x != x || x <= 0.0) return 0;
    if (x >= 18446744073709551616.0) return UINT64_MAX;
    return (uint64_t)x;
}
// f32::max / f32::min -> libm fmaxf/fminf: a NaN operand loses
static inline float rust_maxf(float a, float b) { return (a != a) ? b : (b != b) ? a : (a > b ? a : b); }
static inline float rust_minf(float a, float b) { return (a != a) ? b : (b != b) ? a : (a < b ? a : b); }

// ---------------------------------------------------------------- math (lc3o_math.cpp)
float msun_powf(float x, float y);
float msun_log2f(float x);
float msun_log10f(float x);
float msun_exp2f(float x);
float msun_asinf(float x);
float msun_sinf(float x);
float nt_powi(float base, int32_t exp);   // num_traits no_std powi: recip + square-and-multiply
float fastmath_exp2_raw(float x);         // fast-math 0.1.1 exp2_raw

// ---------------------------------------------------------------- transform substrate
struct Cpx { float r, i; };
static inline Cpx cmul(Cpx a, Cpx b) { return {a.r * b.r - a.i * b.i, a.r * b.i + a.i * b.r}; }
static inline Cpx cadd(Cpx a, Cpx b) { return {a.r + b.r, a.i + b.i}; }
static inline Cpx csub(Cpx a, Cpx b) { return {a.r - b.r, a.i - b.i}; }

// common/kissfft.rs:9-289
struct KissFft {
    int nfft = 0;
    bool inverse = false;
    std::vector<Cpx> twiddle;
    int factors[64] = {0};
    void init(int n, bool inv);
    void transform(const Cpx* fin, Cpx* fout) const;
  private:
    void work(Cpx* fout, const Cpx* fin, int fstride, int in_stride, int factor_idx, int fin_idx,
              int fout_idx) const;
    void bfly2(Cpx* f, int fstride, int m) const;
    void bfly3(Cpx* f, int fstride, int m) const;
    void bfly4(Cpx* f, int fstride, int m) const;
    void bfly5(Cpx* f, int fstride, int m) const;
    void bfly_generic(Cpx* f, int fstride, int m, int p) const;
};

// common/dct_iv.rs:14-72
struct DctIv {
    int nf = 0;
    KissFft fft;
    std::vector<Cpx> input, output, twiddle;
    void init(int nf);
    void run(float* buf);
};

// ---------------------------------------------------------------- decoder (lc3o_decoder.cpp)
struct BufferReader {          // decoder/buffer_reader.rs:12
    int64_t head_byte_cursor = 0, tail_bit_cursor = 0;
    bool read_head_byte(const uint8_t* buf, int64_t len, uint8_t* out);
    bool read_head_u24(const uint8_t* buf, int64_t len, uint32_t* out);
    bool read_tail_usize(const uint8_t* buf, int64_t len, int num_bits, uint64_t* out);
    bool read_tail_bool(const uint8_t* buf, int64_t len, bool* out);
};

struct LtpfInfo { bool pitch_present = false, is_active = false; int pitch_index = 0; };
struct SnsVq { int ind_lf, ind_hf, ls_inda, ls_indb, idx_a, idx_b, submode_lsb, submode_msb, g_ind; };
struct SideInfo {              // decoder/side_info.rs:20
    int bandwidth = 0, lastnz = 0;
    bool lsb_mode = false;
    int global_gain_index = 0, num_tns_filters = 0;
    int rc_order_ari_input[2] = {0, 0};
    SnsVq sns_vq{};
    LtpfInfo ltpf{};
    int noise_factor = 0;
};
struct ArithmeticData {        // decoder/arithmetic_codec.rs:100
    int rc_order[2] = {0, 0};
    int rc_i[16] = {0};
    std::vector<uint8_t> residual_bits;
    int32_t noise_filling_seed = 0;
    bool is_zero_frame = false;
    int frame_num_bits = 0;
};

// error codes: 0 = ok, otherwise which reference error variant fired (for diagnostics only;
// the reference collapses every one of them into "conceal", lc3_decoder.rs:138-141)
bool read_side_info(const uint8_t* buf, int64_t len, BufferReader& rd, int fs_ind, int ne, SideInfo* out);
bool arithmetic_decode(const uint8_t* buf, int64_t len, BufferReader& rd, int fs_ind, int ne,
                       const SideInfo& si, FrameDuration n_ms, int32_t* x /*[400]*/, ArithmeticData* out);
void residual_spectrum_decode(bool lsb_mode, const uint8_t* bits, int nbits, float* spec, int ne);
void apply_noise_filling(bool is_zero_frame, int32_t seed, int bandwidth, FrameDuration d, int noise_factor,
                         const int32_t* xi, float* xf, int ne);
void apply_global_gain(int frame_num_bits, int fs_ind, int gg_ind, float* spec, int ne);
void apply_tns_decode(FrameDuration d, int bandwidth, int num_tns_filters, const int* rc_order,
                      const int* rc_i, int n_rc_i, float* spec);
void mpvq_deenum(int dim_in, int k_val_in, int ls_ind, uint32_t mpvq_ind, int32_t* vec_out);
void sns_decode(const Config& c, const SnsVq& sns, float* spec);
void scale_and_round(const float* x, int n, int16_t* out);

struct Plc {                   // decoder/packet_loss_concealment.rs:7
    std::vector<float> last_good;
    uint64_t num_lost_frames = 0;
    float alpha = 1.0f;
    uint64_t plc_seed = 24607;
    int ne = 0;
    void init(int ne_) { ne = ne_; last_good.assign(ne_, 0.0f); }
    void save(const float* spec);
    LtpfInfo load_into(float* spec, int n);
};

// The CUDA engine's inverse MDCT (lc3o_engine_imdct.cpp): its DCT-IV (lc3b_imdct.cuh's Stockham FFT, not kissfft), its
// unfold and its folded window, tables as the engine builds them.  Opt-in per decoder (TRANSFORM_ENGINE below).
struct EngineImdct {
    int nf = 0, z = 0, n_stages = 0, radices[4] = {0, 0, 0, 0};
    std::vector<Cpx> dtw, ftw;   // DCT-IV pre/post twiddles and FFT twiddles, nf / 2 each
    std::vector<float> win;      // win[m] = gain * w[2 nf - 1 - m], 2 nf
    std::vector<float> p, q;     // the two Stockham buffers
    static bool plan(int n, int* radices, int* count);
    void init(const Config& c);
    void dct_iv(float* buf);     // nf floats in place
    void unfold(const float* D, float* head /*nf*/, float* tail /*nf - z*/) const;
};

// which inverse transform a decoder runs: the reference's (kissfft DCT-IV, gain then window) or the engine's
enum { TRANSFORM_REFERENCE = 0, TRANSFORM_ENGINE = 1 };

struct DecMdct {               // decoder/modified_dct.rs:13
    Config cfg{};
    DctIv dct;
    int transform = TRANSFORM_REFERENCE;
    EngineImdct eng;
    std::vector<float> mem_ola_add, t_hat;
    void init(const Config& c, int transform = TRANSFORM_REFERENCE);
    void run(const float* spec, float* freq);
};

struct DecLtpf {               // decoder/long_term_post_filter.rs:12
    Config cfg{};
    int num_mem_blocks = 0, norm = 0, l_num = 0, l_den = 0;
    bool ltpf_active_prev = false;
    int block_start_index = 0;
    std::vector<float> c_num, c_den, c_num_mem, c_den_mem, x_hat_ltpf_mem, x_hat_mem, scratch;
    int p_int_mem = 0, p_fr_mem = 0;
    void init(const Config& c);
    void run(const LtpfInfo& info, int nbits, float* freq);
  private:
    int wrap(int idx) const;
    float filt(int start, int pitch_int, const std::vector<float>& cn, const std::vector<float>& cd) const;
};

struct DecoderChannel {        // decoder/lc3_decoder.rs:62
    Config cfg{};
    std::vector<float> spec, freq;
    Plc plc;
    DecMdct mdct;
    DecLtpf ltpf;
    uint64_t frame_index = 0;
    // diagnostics of the last frame (what the parity gates compare)
    bool last_ok = false;
    SideInfo last_si{};
    ArithmeticData last_ad{};
    int32_t last_x[400] = {0};
    void init(SamplingFrequency sf, FrameDuration fd, int transform = TRANSFORM_REFERENCE);
    // returns 0, or 1 for Only16BitsPerAudioSampleSupported (lc3_decoder.rs:80)
    int decode(int bits_per_sample, const uint8_t* buf, int64_t len, int16_t* out, int n_out);
};

// ---------------------------------------------------------------- encoder (lc3o_encoder.cpp)
struct EncMdct {               // encoder/modified_dct.rs:18
    Config cfg{};
    DctIv dct;
    std::vector<int16_t> tbuf;   // `freq` in the reference: 2*nf time samples
    void init(const Config& c);
    bool run(const int16_t* in, float* out /*nf*/, float* e_b /*nb*/);
};
struct BwResult { int bandwidth_ind, nbits_bandwidth; };
BwResult bandwidth_detect(const Config& c, const float* e_b);
struct AttackDetector {        // encoder/attack_detector.rs:10
    Config cfg{};
    int num_downsampled = 0, num_blocks = 0, attack_pos_limit = 0;
    float energy_last = 0, max_energy_last = 0;
    int attack_pos_last = -1, tm1 = 0, tm2 = 0;
    void init(const Config& c);
    bool run(const int16_t* x, int nbytes);
};
struct SnsResult { int ind_lf, ind_hf, shape_j, gind, ls_inda, ls_indb; uint64_t index_joint_j; };
SnsResult sns_encode(const Config& c, float* x, const float* e_b, bool attack);
void sns_run_quant(const float* scf, float* scfq, SnsResult* r);
struct TnsResult {
    int nbits_tns, lpc_weighting, num_tns_filters;
    int rc_order[2];
    int rc_i[16];
    float rc_q[16];
};
TnsResult tns_encode(const Config& c, float* x, int p_bw, int nbits, bool near_nyquist);
struct EncLtpfResult { int pitch_index; bool pitch_present, ltpf_active; int nbits_ltpf; };
struct EncLtpf {               // encoder/long_term_post_filter.rs:23
    Config cfg{};
    int len12p8 = 0, len6p4 = 0, delay = 0, up = 0;
    float resamp_fac = 0;
    int t_prev = 17;
    float mem_pitch = 0, mem_nc = 0, mem_mem_nc = 0;
    bool mem_ltpf_active = false;
    std::vector<int16_t> x_s_ext;
    std::vector<float> x12, x6;
    float h50_m1 = 0, h50_m2 = 0;
    void init(const Config& c);
    EncLtpfResult run(const int16_t* x, bool near_nyquist, int nbits);
};
struct QuantResult {
    int gg_ind, nbits_spec, nbits_lsb, nbits_trunc;
    bool lsb_mode;
    int rate_flag, lastnz_trunc;
    float gg;
};
struct SpecQuant {             // encoder/spectral_quantization.rs:50
    int ne = 0, fs_ind = 0;
    bool reset_offset_old = false;
    float nbits_offset_old = 0;
    int nbits_spec_old = 0, nbits_est_old = 0;
    void init(int ne_, int fs_ind_) { ne = ne_; fs_ind = fs_ind_; }
    QuantResult run(const float* x_f, int16_t* x_q, int nbits, int nbits_bw, int nbits_tns, int nbits_ltpf);
};
int residual_encode(int nbits_spec, int nbits_trunc, int ne, float gg, const float* xf, const int16_t* xq,
                    uint8_t* bits /*[400]*/);
int noise_factor(const Config& c, const float* xf, const int16_t* xq, int bw_ind, float gg);
void bitstream_encode(const Config& c, const BwResult& bw, const SnsResult& sns, const TnsResult& tns,
                      const EncLtpfResult& pf, const QuantResult& q, const uint8_t* res_bits, int n_res,
                      int nf_factor, const int16_t* xq, uint8_t* out, int nbytes);

struct EncoderChannel {        // encoder/lc3_encoder.rs:42
    Config cfg{};
    EncMdct mdct;
    AttackDetector attack;
    EncLtpf ltpf;
    SpecQuant quant;
    std::vector<float> mdct_out, e_b;
    std::vector<int16_t> xq;
    uint64_t frame_index = 0;
    void init(SamplingFrequency sf, FrameDuration fd);
    void encode(const int16_t* x, uint8_t* out, int nbytes);
};

}  // namespace lc3o
