// CPU ORACLE - TEST INFRASTRUCTURE (see lc3o.h).
// extern "C" surface for ctypes (oracle/pyoracle.py): stage-level entry points used by the
// golden-vector tests, whole-channel objects, and multi-threaded whole-corpus drivers used
// to build test corpora and to time the CPU baseline.
#include <thread>

#include "lc3o.h"

using namespace lc3o;
namespace lc3o { extern thread_local int g_fail_line; }

// Per-frame inspection record shared with the CUDA engine (include/lc3b.h: LC3B_TRACE_*).
enum {
    TR_OK = 0, TR_BW, TR_LASTNZ, TR_LSB_MODE, TR_GG_IND, TR_NUM_TNS, TR_RC_ORDER_IN0, TR_RC_ORDER_IN1,
    TR_IND_LF, TR_IND_HF, TR_LS_INDA, TR_LS_INDB, TR_IDX_A, TR_IDX_B, TR_SUBMODE_LSB, TR_SUBMODE_MSB, TR_G_IND,
    TR_PITCH_PRESENT, TR_LTPF_ACTIVE, TR_PITCH_INDEX, TR_NOISE_FACTOR, TR_RC_ORDER0, TR_RC_ORDER1,
    TR_RC_I0 /* 16 */, TR_NRES = TR_RC_I0 + 16, TR_SEED, TR_IS_ZERO, TR_WORDS = 48
};

static void fill_trace(const DecoderChannel& ch, int32_t* tr, int32_t* x_out, int ne) {
    for (int i = 0; i < TR_WORDS; i++) tr[i] = 0;
    tr[TR_OK] = ch.last_ok;
    if (ch.last_ok) {
        const SideInfo& s = ch.last_si;
        const ArithmeticData& a = ch.last_ad;
        tr[TR_BW] = s.bandwidth; tr[TR_LASTNZ] = s.lastnz; tr[TR_LSB_MODE] = s.lsb_mode; tr[TR_GG_IND] = s.global_gain_index;
        tr[TR_NUM_TNS] = s.num_tns_filters; tr[TR_RC_ORDER_IN0] = s.rc_order_ari_input[0];
        tr[TR_RC_ORDER_IN1] = s.rc_order_ari_input[1];
        tr[TR_IND_LF] = s.sns_vq.ind_lf; tr[TR_IND_HF] = s.sns_vq.ind_hf; tr[TR_LS_INDA] = s.sns_vq.ls_inda;
        tr[TR_LS_INDB] = s.sns_vq.ls_indb; tr[TR_IDX_A] = s.sns_vq.idx_a; tr[TR_IDX_B] = s.sns_vq.idx_b;
        tr[TR_SUBMODE_LSB] = s.sns_vq.submode_lsb; tr[TR_SUBMODE_MSB] = s.sns_vq.submode_msb; tr[TR_G_IND] = s.sns_vq.g_ind;
        tr[TR_PITCH_PRESENT] = s.ltpf.pitch_present; tr[TR_LTPF_ACTIVE] = s.ltpf.is_active;
        tr[TR_PITCH_INDEX] = s.ltpf.pitch_index; tr[TR_NOISE_FACTOR] = s.noise_factor;
        tr[TR_RC_ORDER0] = a.rc_order[0]; tr[TR_RC_ORDER1] = a.rc_order[1];
        for (int i = 0; i < 16; i++) tr[TR_RC_I0 + i] = a.rc_i[i];
        tr[TR_NRES] = (int32_t)a.residual_bits.size(); tr[TR_SEED] = a.noise_filling_seed; tr[TR_IS_ZERO] = a.is_zero_frame;
    }
    if (x_out) for (int k = 0; k < ne; k++) x_out[k] = ch.last_ok ? ch.last_x[k] : 0;
}

template <class F>
static void parallel_for(int nthreads, int n, F f) {
    if (nthreads <= 1 || n <= 1) { for (int i = 0; i < n; i++) f(i); return; }
    std::vector<std::thread> th;
    for (int t = 0; t < nthreads; t++)
        th.emplace_back([=]() { for (int i = t; i < n; i += nthreads) f(i); });
    for (auto& t : th) t.join();
}

extern "C" {

int lc3o_trace_words() { return TR_WORDS; }
int lc3o_last_fail_line() { return lc3o::g_fail_line; }

void lc3o_config(int sf, int fd, int32_t* out7) {
    Config c = make_config((SamplingFrequency)sf, (FrameDuration)fd);
    out7[0] = c.fs_ind; out7[1] = c.fs; out7[2] = c.ne; out7[3] = c.nb; out7[4] = c.nf; out7[5] = c.z; out7[6] = c.n_ms;
}

// ---------------------------------------------------------------- math
float lc3o_powf(float x, float y) { return msun_powf(x, y); }
float lc3o_log2f(float x) { return msun_log2f(x); }
float lc3o_log10f(float x) { return msun_log10f(x); }
float lc3o_exp2f(float x) { return msun_exp2f(x); }
float lc3o_asinf(float x) { return msun_asinf(x); }
float lc3o_sinf(float x) { return msun_sinf(x); }
float lc3o_powi(float x, int n) { return nt_powi(x, n); }
float lc3o_exp2_raw(float x) { return fastmath_exp2_raw(x); }
void lc3o_math_vec(int which, const float* x, const float* y, float* out, int n) {
    for (int i = 0; i < n; i++) {
        switch (which) {
            case 0: out[i] = msun_powf(x[i], y[i]); break;
            case 1: out[i] = msun_log2f(x[i]); break;
            case 2: out[i] = msun_log10f(x[i]); break;
            case 3: out[i] = msun_exp2f(x[i]); break;
            case 4: out[i] = msun_asinf(x[i]); break;
            case 5: out[i] = msun_sinf(x[i]); break;
            case 6: out[i] = fastmath_exp2_raw(x[i]); break;
        }
    }
}

// ---------------------------------------------------------------- transforms
void lc3o_kissfft(int n, const float* in_r, const float* in_i, float* out_r, float* out_i) {
    KissFft k;
    k.init(n, false);
    std::vector<Cpx> fin(n), fout(n);
    for (int i = 0; i < n; i++) fin[i] = {in_r[i], in_i[i]};
    k.transform(fin.data(), fout.data());
    for (int i = 0; i < n; i++) { out_r[i] = fout[i].r; out_i[i] = fout[i].i; }
}
void lc3o_kissfft_factors(int n, int32_t* out64) {
    KissFft k;
    k.init(n, false);
    for (int i = 0; i < 64; i++) out64[i] = k.factors[i];
}
void lc3o_dct_iv(int nf, float* buf) {
    DctIv d;
    d.init(nf);
    d.run(buf);
}

// the decoder's MDCT window w_N (2 nf entries, decoder/modified_dct.rs:37-56)
void lc3o_mdct_window(int sf, int fd, float* out) {
    Config c = make_config((SamplingFrequency)sf, (FrameDuration)fd);
    std::memcpy(out, mdct_window(c), sizeof(float) * 2 * c.nf);
}

// the engine's inverse MDCT pieces (lc3o_engine_imdct.cpp) for the configuration (sf, fd)
void lc3o_engine_dct_iv(int sf, int fd, float* buf) {
    EngineImdct e;
    e.init(make_config((SamplingFrequency)sf, (FrameDuration)fd));
    e.dct_iv(buf);
}
void lc3o_engine_unfold(int sf, int fd, const float* D, float* head, float* tail) {
    EngineImdct e;
    e.init(make_config((SamplingFrequency)sf, (FrameDuration)fd));
    e.unfold(D, head, tail);
}
// win [2 nf], dtw and ftw [nf / 2][2]
void lc3o_engine_tables(int sf, int fd, float* win, float* dtw, float* ftw) {
    EngineImdct e;
    e.init(make_config((SamplingFrequency)sf, (FrameDuration)fd));
    for (int m = 0; m < 2 * e.nf; m++) win[m] = e.win[m];
    for (int i = 0; i < e.nf / 2; i++) {
        dtw[2 * i] = e.dtw[i].r; dtw[2 * i + 1] = e.dtw[i].i;
        ftw[2 * i] = e.ftw[i].r; ftw[2 * i + 1] = e.ftw[i].i;
    }
}

// ---------------------------------------------------------------- decoder stages
int lc3o_read_tail_usize(const uint8_t* buf, int len, int head, int* tail_cursor, int nbits, uint64_t* out) {
    BufferReader r;
    r.head_byte_cursor = head;
    r.tail_bit_cursor = *tail_cursor;
    bool ok = r.read_tail_usize(buf, len, nbits, out);
    *tail_cursor = (int)r.tail_bit_cursor;
    return ok;
}
int lc3o_read_tail_bool(const uint8_t* buf, int len, int head, int* tail_cursor, int* out) {
    BufferReader r;
    r.head_byte_cursor = head;
    r.tail_bit_cursor = *tail_cursor;
    bool b = false;
    bool ok = r.read_tail_bool(buf, len, &b);
    *tail_cursor = (int)r.tail_bit_cursor;
    *out = b;
    return ok;
}

static void si_to_arr(const SideInfo& s, int32_t* o) {
    o[0] = s.bandwidth; o[1] = s.lastnz; o[2] = s.lsb_mode; o[3] = s.global_gain_index; o[4] = s.num_tns_filters;
    o[5] = s.rc_order_ari_input[0]; o[6] = s.rc_order_ari_input[1];
    o[7] = s.sns_vq.ind_lf; o[8] = s.sns_vq.ind_hf; o[9] = s.sns_vq.ls_inda; o[10] = s.sns_vq.ls_indb;
    o[11] = s.sns_vq.idx_a; o[12] = s.sns_vq.idx_b; o[13] = s.sns_vq.submode_lsb; o[14] = s.sns_vq.submode_msb;
    o[15] = s.sns_vq.g_ind; o[16] = s.ltpf.pitch_present; o[17] = s.ltpf.is_active; o[18] = s.ltpf.pitch_index;
    o[19] = s.noise_factor;
}
static SideInfo arr_to_si(const int32_t* o) {
    SideInfo s;
    s.bandwidth = o[0]; s.lastnz = o[1]; s.lsb_mode = o[2]; s.global_gain_index = o[3]; s.num_tns_filters = o[4];
    s.rc_order_ari_input[0] = o[5]; s.rc_order_ari_input[1] = o[6];
    s.sns_vq = {o[7], o[8], o[9], o[10], o[11], o[12], o[13], o[14], o[15]};
    s.ltpf.pitch_present = o[16]; s.ltpf.is_active = o[17]; s.ltpf.pitch_index = o[18];
    s.noise_factor = o[19];
    return s;
}

// out20: the SideInfo fields in si_to_arr order; returns 1 on Ok; *tail_cursor = bits consumed
int lc3o_read_side_info(const uint8_t* buf, int len, int fs_ind, int ne, int32_t* out20, int* tail_cursor) {
    BufferReader r;
    SideInfo s;
    bool ok = read_side_info(buf, len, r, fs_ind, ne, &s);
    if (ok) si_to_arr(s, out20);
    *tail_cursor = (int)r.tail_bit_cursor;
    return ok;
}

// out_misc: [rc_order0, rc_order1, n_residual_bits, seed, is_zero_frame, frame_num_bits]
int lc3o_arithmetic_decode(const uint8_t* buf, int len, int head, int tail, int fs_ind, int ne, const int32_t* si20,
                           int n_ms, int32_t* x400, int32_t* rc_i16, uint8_t* res_bits480, int32_t* out_misc) {
    BufferReader r;
    r.head_byte_cursor = head;
    r.tail_bit_cursor = tail;
    SideInfo s = arr_to_si(si20);
    ArithmeticData a;
    for (int i = 0; i < 400; i++) x400[i] = 0;
    bool ok = arithmetic_decode(buf, len, r, fs_ind, ne, s, (FrameDuration)n_ms, x400, &a);
    if (!ok) return 0;
    for (int i = 0; i < 16; i++) rc_i16[i] = a.rc_i[i];
    for (size_t i = 0; i < a.residual_bits.size(); i++) res_bits480[i] = a.residual_bits[i];
    out_misc[0] = a.rc_order[0]; out_misc[1] = a.rc_order[1]; out_misc[2] = (int32_t)a.residual_bits.size();
    out_misc[3] = a.noise_filling_seed; out_misc[4] = a.is_zero_frame; out_misc[5] = a.frame_num_bits;
    return 1;
}

void lc3o_residual_spectrum_decode(int lsb_mode, const uint8_t* bits, int nbits, float* spec, int ne) {
    residual_spectrum_decode(lsb_mode, bits, nbits, spec, ne);
}
void lc3o_noise_filling(int is_zero, int seed, int bw, int n_ms, int nf_factor, const int32_t* xi, float* xf, int ne) {
    apply_noise_filling(is_zero, seed, bw, (FrameDuration)n_ms, nf_factor, xi, xf, ne);
}
void lc3o_global_gain(int nbits, int fs_ind, int gg_ind, float* spec, int n) { apply_global_gain(nbits, fs_ind, gg_ind, spec, n); }
void lc3o_tns_decode(int n_ms, int bw, int num_filters, const int32_t* rc_order, const int32_t* rc_i, int n_rc_i, float* spec) {
    int o[2] = {rc_order[0], rc_order[1]}, ri[16] = {0};
    for (int i = 0; i < n_rc_i && i < 16; i++) ri[i] = rc_i[i];
    apply_tns_decode((FrameDuration)n_ms, bw, num_filters, o, ri, n_rc_i, spec);
}
void lc3o_mpvq_deenum(int dim, int k, int ls_ind, uint32_t idx, int32_t* out16) { mpvq_deenum(dim, k, ls_ind, idx, out16); }
void lc3o_sns_decode(int sf, int fd, const int32_t* sns9, float* spec) {
    Config c = make_config((SamplingFrequency)sf, (FrameDuration)fd);
    SnsVq s = {sns9[0], sns9[1], sns9[2], sns9[3], sns9[4], sns9[5], sns9[6], sns9[7], sns9[8]};
    sns_decode(c, s, spec);
}
void lc3o_scale_and_round(const float* x, int n, int16_t* out) { scale_and_round(x, n, out); }

// PLC object
void* lc3o_plc_new(int ne) { Plc* p = new Plc; p->init(ne); return p; }
void lc3o_plc_save(void* h, const float* spec) { ((Plc*)h)->save(spec); }
void lc3o_plc_load(void* h, float* spec, int n) { ((Plc*)h)->load_into(spec, n); }
void lc3o_plc_free(void* h) { delete (Plc*)h; }

// decoder MDCT object
void* lc3o_decmdct_new(int sf, int fd) { DecMdct* m = new DecMdct; m->init(make_config((SamplingFrequency)sf, (FrameDuration)fd)); return m; }
void* lc3o_decmdct_new_ex(int sf, int fd, int transform) {
    DecMdct* m = new DecMdct;
    m->init(make_config((SamplingFrequency)sf, (FrameDuration)fd), transform);
    return m;
}
void lc3o_decmdct_run(void* h, const float* spec, float* freq) { ((DecMdct*)h)->run(spec, freq); }
void lc3o_decmdct_free(void* h) { delete (DecMdct*)h; }

// decoder LTPF object
void* lc3o_decltpf_new(int sf, int fd) { DecLtpf* m = new DecLtpf; m->init(make_config((SamplingFrequency)sf, (FrameDuration)fd)); return m; }
void lc3o_decltpf_run(void* h, int is_active, int pitch_present, int pitch_index, int nbits, float* freq) {
    LtpfInfo i;
    i.is_active = is_active; i.pitch_present = pitch_present; i.pitch_index = pitch_index;
    ((DecLtpf*)h)->run(i, nbits, freq);
}
void lc3o_decltpf_free(void* h) { delete (DecLtpf*)h; }

// whole decoder channel
void* lc3o_decoder_new(int sf, int fd) { DecoderChannel* d = new DecoderChannel; d->init((SamplingFrequency)sf, (FrameDuration)fd); return d; }
void lc3o_decoder_free(void* h) { delete (DecoderChannel*)h; }
int lc3o_decoder_decode(void* h, int bits_per_sample, const uint8_t* buf, int len, int16_t* out, int n_out,
                        int32_t* trace /*nullable*/, int32_t* x_out /*nullable*/) {
    DecoderChannel* d = (DecoderChannel*)h;
    int rc = d->decode(bits_per_sample, buf, len, out, n_out);
    if (rc == 0 && trace) fill_trace(*d, trace, x_out, d->cfg.ne);
    return rc;
}

// ---------------------------------------------------------------- encoder stages
void* lc3o_encmdct_new(int sf, int fd) { EncMdct* m = new EncMdct; m->init(make_config((SamplingFrequency)sf, (FrameDuration)fd)); return m; }
int lc3o_encmdct_run(void* h, const int16_t* in, float* out, float* e_b) { return ((EncMdct*)h)->run(in, out, e_b); }
void lc3o_encmdct_free(void* h) { delete (EncMdct*)h; }

void lc3o_bandwidth_detect(int sf, int fd, const float* e_b, int32_t* out2) {
    BwResult r = bandwidth_detect(make_config((SamplingFrequency)sf, (FrameDuration)fd), e_b);
    out2[0] = r.bandwidth_ind; out2[1] = r.nbits_bandwidth;
}

void* lc3o_attack_new(int sf, int fd) { AttackDetector* a = new AttackDetector; a->init(make_config((SamplingFrequency)sf, (FrameDuration)fd)); return a; }
int lc3o_attack_run(void* h, const int16_t* x, int nbytes) { return ((AttackDetector*)h)->run(x, nbytes); }
void lc3o_attack_state(void* h, float* f2, int32_t* i4) {
    AttackDetector* a = (AttackDetector*)h;
    f2[0] = a->max_energy_last; f2[1] = a->energy_last;
    i4[0] = a->num_downsampled; i4[1] = a->attack_pos_last; i4[2] = a->tm1; i4[3] = a->tm2;
}
void lc3o_attack_free(void* h) { delete (AttackDetector*)h; }

static void sns_to_arr(const SnsResult& r, int64_t* o) {
    o[0] = r.ind_lf; o[1] = r.ind_hf; o[2] = r.shape_j; o[3] = r.gind; o[4] = r.ls_inda; o[5] = r.ls_indb; o[6] = (int64_t)r.index_joint_j;
}
void lc3o_sns_encode(int sf, int fd, float* x, const float* e_b, int attack, int64_t* out7) {
    SnsResult r = sns_encode(make_config((SamplingFrequency)sf, (FrameDuration)fd), x, e_b, attack);
    sns_to_arr(r, out7);
}
void lc3o_sns_quant(const float* scf, float* scfq, int64_t* out7) {
    SnsResult r{};
    sns_run_quant(scf, scfq, &r);
    sns_to_arr(r, out7);
}
// out_i: [nbits_tns, lpc_weighting, num_tns_filters, rc_order0, rc_order1, rc_i[16]]
void lc3o_tns_encode(int sf, int fd, float* x, int p_bw, int nbits, int near_nyquist, int32_t* out_i21, float* rc_q16) {
    TnsResult r = tns_encode(make_config((SamplingFrequency)sf, (FrameDuration)fd), x, p_bw, nbits, near_nyquist);
    out_i21[0] = r.nbits_tns; out_i21[1] = r.lpc_weighting; out_i21[2] = r.num_tns_filters;
    out_i21[3] = r.rc_order[0]; out_i21[4] = r.rc_order[1];
    for (int i = 0; i < 16; i++) { out_i21[5 + i] = r.rc_i[i]; rc_q16[i] = r.rc_q[i]; }
}
void* lc3o_encltpf_new(int sf, int fd) { EncLtpf* m = new EncLtpf; m->init(make_config((SamplingFrequency)sf, (FrameDuration)fd)); return m; }
void lc3o_encltpf_run(void* h, const int16_t* x, int near_nyquist, int nbits, int32_t* out4) {
    EncLtpfResult r = ((EncLtpf*)h)->run(x, near_nyquist, nbits);
    out4[0] = r.pitch_index; out4[1] = r.pitch_present; out4[2] = r.ltpf_active; out4[3] = r.nbits_ltpf;
}
void lc3o_encltpf_free(void* h) { delete (EncLtpf*)h; }

void* lc3o_quant_new(int ne, int fs_ind) { SpecQuant* q = new SpecQuant; q->init(ne, fs_ind); return q; }
// out_i: [gg_ind, nbits_spec, nbits_lsb, nbits_trunc, lsb_mode, rate_flag, lastnz_trunc]
void lc3o_quant_run(void* h, const float* xf, int16_t* xq, int nbits, int nbits_bw, int nbits_tns, int nbits_ltpf,
                    int32_t* out_i7, float* gg) {
    QuantResult r = ((SpecQuant*)h)->run(xf, xq, nbits, nbits_bw, nbits_tns, nbits_ltpf);
    out_i7[0] = r.gg_ind; out_i7[1] = r.nbits_spec; out_i7[2] = r.nbits_lsb; out_i7[3] = r.nbits_trunc;
    out_i7[4] = r.lsb_mode; out_i7[5] = r.rate_flag; out_i7[6] = r.lastnz_trunc;
    *gg = r.gg;
}
void lc3o_quant_free(void* h) { delete (SpecQuant*)h; }

int lc3o_noise_factor(int sf, int fd, const float* xf, const int16_t* xq, int bw, float gg) {
    return noise_factor(make_config((SamplingFrequency)sf, (FrameDuration)fd), xf, xq, bw, gg);
}

// bitstream_encode with every input spelled out (bitstream_encoding.rs::bitstream_encoding_run)
void lc3o_bitstream_encode(int sf, int fd, int bw_ind, int nbits_bw, const int64_t* sns7, int lpc_weighting,
                           int num_tns_filters, const int32_t* rc_order2, const int32_t* rc_i16, int pitch_present,
                           int ltpf_active, int pitch_index, int gg_ind, int lsb_mode, int rate_flag, int lastnz_trunc,
                           int nbits_lsb, const uint8_t* res_bits, int n_res, int nf_factor, const int16_t* xq,
                           uint8_t* out, int nbytes) {
    Config c = make_config((SamplingFrequency)sf, (FrameDuration)fd);
    BwResult bw{bw_ind, nbits_bw};
    SnsResult s{(int)sns7[0], (int)sns7[1], (int)sns7[2], (int)sns7[3], (int)sns7[4], (int)sns7[5], (uint64_t)sns7[6]};
    TnsResult t{};
    t.lpc_weighting = lpc_weighting; t.num_tns_filters = num_tns_filters;
    t.rc_order[0] = rc_order2[0]; t.rc_order[1] = rc_order2[1];
    for (int i = 0; i < 16; i++) t.rc_i[i] = rc_i16[i];
    EncLtpfResult p{pitch_index, pitch_present != 0, ltpf_active != 0, pitch_present ? 11 : 1};
    QuantResult q{};
    q.gg_ind = gg_ind; q.lsb_mode = lsb_mode; q.rate_flag = rate_flag; q.lastnz_trunc = lastnz_trunc; q.nbits_lsb = nbits_lsb;
    bitstream_encode(c, bw, s, t, p, q, res_bits, n_res, nf_factor, xq, out, nbytes);
}

// whole encoder channel
void* lc3o_encoder_new(int sf, int fd) { EncoderChannel* e = new EncoderChannel; e->init((SamplingFrequency)sf, (FrameDuration)fd); return e; }
void lc3o_encoder_free(void* h) { delete (EncoderChannel*)h; }
void lc3o_encoder_encode(void* h, const int16_t* x, uint8_t* out, int nbytes) { ((EncoderChannel*)h)->encode(x, out, nbytes); }

// ---------------------------------------------------------------- whole-corpus drivers
// Layouts: pcm [n_streams][n_frames][nf] i16, bytes [n_streams][n_frames][nbytes] u8.
// nbytes_per_frame: optional [n_streams][n_frames] i32; 0 = frame lost (decoder is handed an empty buffer,
// which the reference turns into concealment because the first tail read fails).
void lc3o_encode_streams(int nthreads, int n_streams, int n_frames, const int32_t* sf_fd /*[n_streams][2] or null*/,
                         int sf, int fd, const int16_t* pcm, int nf_stride, uint8_t* bytes, int nbytes) {
    parallel_for(nthreads, n_streams, [=](int s) {
        int ssf = sf_fd ? sf_fd[2 * s] : sf, sfd = sf_fd ? sf_fd[2 * s + 1] : fd;
        EncoderChannel e;
        e.init((SamplingFrequency)ssf, (FrameDuration)sfd);
        for (int f = 0; f < n_frames; f++)
            e.encode(pcm + ((size_t)s * n_frames + f) * nf_stride, bytes + ((size_t)s * n_frames + f) * nbytes, nbytes);
    });
}

// transform: TRANSFORM_REFERENCE (the reference's kissfft DCT-IV) or TRANSFORM_ENGINE (the CUDA engine's inverse MDCT)
void lc3o_decode_streams_ex(int nthreads, int n_streams, int n_frames, int sf, int fd, const uint8_t* bytes, int nbytes,
                            const int32_t* nbytes_per_frame /*nullable*/, int16_t* pcm, int32_t* trace /*nullable*/,
                            int32_t* x_out /*nullable*/, float* spec_out /*nullable: spectrum handed to the IMDCT*/,
                            int transform) {
    Config c = make_config((SamplingFrequency)sf, (FrameDuration)fd);
    parallel_for(nthreads, n_streams, [=](int s) {
        DecoderChannel d;
        d.init((SamplingFrequency)sf, (FrameDuration)fd, transform);
        for (int f = 0; f < n_frames; f++) {
            size_t fi = (size_t)s * n_frames + f;
            int len = nbytes_per_frame ? nbytes_per_frame[fi] : nbytes;
            d.decode(16, bytes + fi * nbytes, len, pcm + fi * c.nf, c.nf);
            if (trace) fill_trace(d, trace + fi * TR_WORDS, x_out ? x_out + fi * c.ne : nullptr, c.ne);
            if (spec_out) std::memcpy(spec_out + fi * c.ne, d.spec.data(), sizeof(float) * c.ne);
        }
    });
}
void lc3o_decode_streams(int nthreads, int n_streams, int n_frames, int sf, int fd, const uint8_t* bytes, int nbytes,
                         const int32_t* nbytes_per_frame /*nullable*/, int16_t* pcm, int32_t* trace /*nullable*/,
                         int32_t* x_out /*nullable*/, float* spec_out /*nullable: spectrum handed to the IMDCT*/) {
    lc3o_decode_streams_ex(nthreads, n_streams, n_frames, sf, fd, bytes, nbytes, nbytes_per_frame, pcm, trace, x_out,
                           spec_out, TRANSFORM_REFERENCE);
}

}  // extern "C"
