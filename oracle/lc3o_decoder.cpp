// CPU ORACLE - TEST INFRASTRUCTURE (see lc3o.h).
// Decoder restatement: src/decoder/*.rs of the reference, stage by stage, quirks included.
#include "lc3o.h"

namespace lc3o {

// diagnostics only: source line of the last decode error on this thread (which reference error variant fired)
thread_local int g_fail_line = 0;
#define FAIL() (g_fail_line = __LINE__, false)

// ================================================================== buffer_reader.rs
// buffer_reader.rs:42-50
bool BufferReader::read_head_byte(const uint8_t* buf, int64_t len, uint8_t* out) {
    if (head_byte_cursor < len) { *out = buf[head_byte_cursor++]; return true; }
    return FAIL();
}
// buffer_reader.rs:52-60
bool BufferReader::read_head_u24(const uint8_t* buf, int64_t len, uint32_t* out) {
    if (head_byte_cursor + 2 < len) {
        const uint8_t* p = buf + head_byte_cursor;
        *out = ((uint32_t)p[0] << 16) | ((uint32_t)p[1] << 8) | p[2];
        head_byte_cursor += 3;
        return true;
    }
    return FAIL();
}
// buffer_reader.rs:63-96: big-endian load of the 1..4 bytes that hold the field, then shifts.
// The bounds test involves the HEAD cursor (tail reads may not cross into consumed head bytes).
bool BufferReader::read_tail_usize(const uint8_t* buf, int64_t len, int num_bits, uint64_t* out) {
    int64_t byte_index = tail_bit_cursor / 8;
    int bit_index = (int)(tail_bit_cursor % 8);
    int bits_left = 8 - bit_index;
    int add_bytes = (num_bits > bits_left && num_bits < 8) ? 2 : 1;
    int num_bytes = num_bits / 8 + add_bytes;
    if ((int32_t)len - (int32_t)head_byte_cursor - (int32_t)byte_index - (int32_t)num_bytes < 0) return FAIL();
    int64_t from = len - byte_index - num_bytes;
    const uint8_t* s = buf + from;
    uint32_t value;
    switch (num_bytes) {
        case 1: value = s[0]; break;
        case 2: value = ((uint32_t)s[0] << 8) | s[1]; break;
        case 3: value = ((uint32_t)s[0] << 16) | ((uint32_t)s[1] << 8) | s[2]; break;
        case 4: value = ((uint32_t)s[0] << 24) | ((uint32_t)s[1] << 16) | ((uint32_t)s[2] << 8) | s[3]; break;
        default: value = 0; break;
    }
    int shift_by = 32 - num_bits - bit_index;
    value <<= shift_by;
    value >>= shift_by + bit_index;
    tail_bit_cursor += num_bits;
    *out = value;
    return true;
}
// buffer_reader.rs:98-114.  QUIRK: the bounds test is looser (+2) than read_tail_usize's.
bool BufferReader::read_tail_bool(const uint8_t* buf, int64_t len, bool* out) {
    int64_t byte_index = tail_bit_cursor / 8;
    int bit_index = (int)(tail_bit_cursor % 8);
    if ((int32_t)len - (int32_t)head_byte_cursor - (int32_t)byte_index + 2 < 0) return FAIL();
    int64_t from = len - byte_index - 1;
    if (from < 0) return FAIL();   // the reference would panic (index out of range); unreachable for nbytes >= 20
    uint8_t byte = buf[from];
    byte = (uint8_t)(byte << (7 - bit_index));
    byte >>= 7;
    tail_bit_cursor += 1;
    *out = byte == 1;
    return true;
}

// ================================================================== side_info_reader.rs
static int lastnz_bits(int ne) {
    // ((ne/2) as f32).log2().ceil(): ne/2 is never a power of two, so this is exact integer work
    int v = ne / 2, b = 0;
    while ((1 << b) < v) b++;
    return b;
}

// side_info_reader.rs:127-200
static bool read_sns_vq(const uint8_t* buf, int64_t len, BufferReader& rd, SnsVq* o) {
    uint64_t v;
    bool b;
    if (!rd.read_tail_usize(buf, len, 5, &v)) return FAIL();
    o->ind_lf = (int)v;
    if (!rd.read_tail_usize(buf, len, 5, &v)) return FAIL();
    o->ind_hf = (int)v;
    if (!rd.read_tail_bool(buf, len, &b)) return FAIL();
    o->submode_msb = b;
    if (!rd.read_tail_usize(buf, len, o->submode_msb == 0 ? 1 : 2, &v)) return FAIL();
    int g_ind = (int)v;
    if (!rd.read_tail_bool(buf, len, &b)) return FAIL();
    o->ls_inda = b;
    if (o->submode_msb == 0) {
        if (!rd.read_tail_usize(buf, len, 25, &v)) return FAIL();
        int64_t tmp = (int64_t)v;
        if (tmp >= 33460056) return FAIL();                     // PlcTriggerSns1OutOfRange
        int64_t idx_bor_gain_lsb = tmp / 2390004;
        o->idx_a = (int)(tmp - idx_bor_gain_lsb * 2390004);
        o->submode_lsb = 0;
        int32_t t = (int32_t)idx_bor_gain_lsb - 2;
        if (t < 0) o->submode_lsb = 1;
        int32_t u = t + o->submode_lsb * 2;
        if (o->submode_lsb != 0) {
            g_ind = (g_ind << 1) + u;
            o->idx_b = 0;
            o->ls_indb = 0;
        } else {
            o->idx_b = u >> 1;
            o->ls_indb = u & 1;
        }
    } else {
        o->ls_indb = 0;
        o->idx_b = 0;
        o->submode_lsb = 0;
        if (!rd.read_tail_usize(buf, len, 24, &v)) return FAIL();
        int64_t tmp = (int64_t)v;
        if (tmp >= 16708096) return FAIL();                     // PlcTriggerSns2OutOfRange
        if (tmp >= 15158272) {
            tmp -= 15158272;
            o->submode_lsb = 1;
            g_ind = (g_ind << 1) + (int)(tmp & 1);
            o->idx_a = (int)(tmp >> 1);
        } else {
            o->idx_a = (int)tmp;
        }
    }
    o->g_ind = g_ind;
    return true;
}

// side_info_reader.rs:29-103
bool read_side_info(const uint8_t* buf, int64_t len, BufferReader& rd, int fs_ind, int ne, SideInfo* o) {
    static const int NBITS_BW_TABLE[5] = {0, 1, 2, 2, 3};
    uint64_t v;
    bool b;
    int nbits_bw = NBITS_BW_TABLE[fs_ind];
    int p_bw = 0;
    if (nbits_bw > 0) {
        if (!rd.read_tail_usize(buf, len, nbits_bw, &v)) return FAIL();
        if ((uint64_t)fs_ind < v) return FAIL();                // BandwidthIdxOutOfRange
        p_bw = (int)v;
    }
    if (!rd.read_tail_usize(buf, len, lastnz_bits(ne), &v)) return FAIL();
    int lastnz = (int)((v + 1) << 1);
    if (lastnz > ne) return FAIL();                             // LastNonZeroTupleGreaterThanYLen
    if (!rd.read_tail_bool(buf, len, &b)) return FAIL();
    o->lsb_mode = b;
    if (!rd.read_tail_usize(buf, len, 8, &v)) return FAIL();
    o->global_gain_index = (int)v;
    o->num_tns_filters = p_bw < 3 ? 1 : 2;
    o->rc_order_ari_input[0] = o->rc_order_ari_input[1] = 0;
    for (int f = 0; f < o->num_tns_filters; f++) {
        if (!rd.read_tail_bool(buf, len, &b)) return FAIL();
        o->rc_order_ari_input[f] = b;
    }
    bool pitch_present;
    if (!rd.read_tail_bool(buf, len, &pitch_present)) return FAIL();
    if (!read_sns_vq(buf, len, rd, &o->sns_vq)) return FAIL();
    // side_info_reader.rs:105-125
    o->ltpf.pitch_present = pitch_present;
    o->ltpf.is_active = false;
    o->ltpf.pitch_index = 0;
    if (pitch_present) {
        if (!rd.read_tail_bool(buf, len, &b)) return FAIL();
        o->ltpf.is_active = b;
        if (!rd.read_tail_usize(buf, len, 9, &v)) return FAIL();
        o->ltpf.pitch_index = (int)v;
    }
    if (!rd.read_tail_usize(buf, len, 3, &v)) return FAIL();
    o->noise_factor = (int)v;
    o->bandwidth = p_bw;   // 0..4 by construction (p_bw <= fs_ind <= 4)
    o->lastnz = lastnz;
    return true;
}

// ================================================================== arithmetic_codec.rs
struct AcState { uint32_t low, range; };

// arithmetic_codec.rs:67-97
static bool ac_decode(const uint8_t* buf, int64_t len, BufferReader& rd, AcState& st, const int16_t* cum,
                      const int16_t* freq, int n_sym, int* out) {
    uint32_t tmp = st.range >> 10;
    uint32_t limit = tmp << 10;
    if (st.low >= limit) return FAIL();                         // AcRangeFlOutOfRange
    int val = n_sym - 1;
    while (st.low < tmp * (uint32_t)(int32_t)cum[val]) val--;
    st.low -= tmp * (uint32_t)(int32_t)cum[val];
    st.range = tmp * (uint32_t)(int32_t)freq[val];
    while (st.range < 0x10000) {
        st.low <<= 8;
        st.low &= 0x00ffffff;
        uint8_t byte;
        if (!rd.read_head_byte(buf, len, &byte)) return FAIL();
        st.low += byte;
        st.range <<= 8;
    }
    *out = val;
    return true;
}

// arithmetic_codec.rs:307-344
static bool decode_tns_data(const uint8_t* buf, int64_t len, BufferReader& rd, const SideInfo& si, AcState& st,
                            int nbits, FrameDuration n_ms, int* tns_idx, int* tns_order) {
    int max_bits = n_ms == SevenPointFiveMs ? 360 : 480;
    int w = nbits < max_bits ? 1 : 0;
    for (int i = 0; i < 16; i++) tns_idx[i] = 0;
    tns_order[0] = si.rc_order_ari_input[0];
    tns_order[1] = si.rc_order_ari_input[1];
    for (int f = 0; f < si.num_tns_filters; f++) {
        if (tns_order[f] > 0) {
            int order;
            if (!ac_decode(buf, len, rd, st, LC3T_AC_TNS_ORDER_CUMFREQ[w], LC3T_AC_TNS_ORDER_FREQ[w], 8, &order))
                return FAIL();
            tns_order[f] = order + 1;
            for (int k = 0; k < tns_order[f]; k++) {
                if (!ac_decode(buf, len, rd, st, LC3T_AC_TNS_COEF_CUMFREQ[k], LC3T_AC_TNS_COEF_FREQ[k], 17,
                               &tns_idx[f * 8 + k]))
                    return FAIL();
            }
        }
    }
    return true;
}

// arithmetic_codec.rs:211-305
static bool decode_spectral_data(const uint8_t* buf, int64_t len, BufferReader& rd, const SideInfo& si, int nbits,
                                 int fs_ind, int ne, AcState& st, int32_t* x, int32_t* save_lev) {
    int rate_flag = nbits > (160 + fs_ind * 160) ? 512 : 0;
    int c = 0;
    for (int k = 0; k < si.lastnz / 2; k++) {
        int t = c + rate_flag + ((k * 2) > (ne / 2) ? 256 : 0);
        int32_t xa = 0, xb = 0;
        int sym = 0, lev = 0;
        bool bit;
        while (lev < 14) {
            int pki = LC3T_AC_SPEC_LOOKUP[t + (lev < 3 ? lev : 3) * 1024];
            if (!ac_decode(buf, len, rd, st, LC3T_AC_SPEC_CUMFREQ[pki], LC3T_AC_SPEC_FREQ[pki], 17, &sym))
                return FAIL();
            if (sym < 16) break;
            if (!si.lsb_mode || lev > 0) {
                if (!rd.read_tail_bool(buf, len, &bit)) return FAIL();
                xa += (int32_t)bit << lev;
                if (!rd.read_tail_bool(buf, len, &bit)) return FAIL();
                xb += (int32_t)bit << lev;
            }
            lev++;
        }
        // QUIRK (i): written by TUPLE index k, later read by LINE index (decode_residual_bits)
        if (si.lsb_mode) save_lev[k] = lev;
        // QUIRK (ii): no lev == 14 bit-error check; sym may be 16 here
        int a = sym & 3, b = sym >> 2;
        xa += (int32_t)a << lev;
        xb += (int32_t)b << lev;
        if (xa > 0) {
            if (!rd.read_tail_bool(buf, len, &bit)) return FAIL();
            if (bit) xa = -xa;
        }
        if (xb > 0) {
            if (!rd.read_tail_bool(buf, len, &bit)) return FAIL();
            if (bit) xb = -xb;
        }
        x[2 * k] = xa;
        x[2 * k + 1] = xb;
        int l = lev < 3 ? lev : 3;
        t = (l <= 1) ? 1 + (a + b) * (l + 1) : 12 + l;
        c = (c & 15) * 16 + t;
    }
    return true;
}

// arithmetic_codec.rs:346-388
static bool read_res_bit(int32_t* x, BufferReader& rd, const uint8_t* buf, int64_t len, int idx, int64_t* nres,
                         bool* cont) {
    if (*nres == 0) { *cont = false; return true; }
    bool bit;
    if (!rd.read_tail_bool(buf, len, &bit)) return FAIL();
    *nres -= 1;
    if (bit) {
        int32_t& v = x[idx];
        if (v > 0) v += 1;
        else if (v < 0) v -= 1;
        else {
            if (*nres == 0) { *cont = false; return true; }
            if (!rd.read_tail_bool(buf, len, &bit)) return FAIL();
            *nres -= 1;
            v = bit ? -1 : 1;
        }
    }
    *cont = true;
    return true;
}

static inline int ilog2_u32(uint32_t v) { return 31 - __builtin_clz(v); }

// arithmetic_codec.rs:109-158
bool arithmetic_decode(const uint8_t* buf, int64_t len, BufferReader& rd, int fs_ind, int ne, const SideInfo& si,
                       FrameDuration n_ms, int32_t* x, ArithmeticData* out) {
    int nbits = (int)len * 8;
    AcState st;
    if (!rd.read_head_u24(buf, len, &st.low)) return FAIL();    // ac_dec_init :57
    st.range = 0x00ffffff;
    if (!decode_tns_data(buf, len, rd, si, st, nbits, n_ms, out->rc_i, out->rc_order)) return FAIL();

    int32_t save_lev[400];
    std::memset(save_lev, 0, sizeof(save_lev));
    if (!decode_spectral_data(buf, len, rd, si, nbits, fs_ind, ne, st, x, save_lev)) return FAIL();
    for (int k = si.lastnz; k < 400; k++) x[k] = 0;            // x is [i32; MAX_LEN_SPECTRAL]

    // decode_residual_bits :160-209 with calc_num_residual_bits :390-407
    int64_t nbits_side = rd.tail_bit_cursor - 8;
    // f64 log2 + floor of an integer in [1, 2^24): exact integer log2.  range == 0 cannot reach here
    // (the renormalisation loop above would have run out of bytes first).
    int64_t nbits_ari = (rd.head_byte_cursor + 1 - 3) * 8 + 25 - (int64_t)ilog2_u32(st.range);
    if ((int64_t)nbits < nbits_side + nbits_ari) return FAIL(); // NegativeResidualNumBits
    int64_t nres = nbits - nbits_side - nbits_ari;
    out->residual_bits.clear();
    if (!si.lsb_mode) {
        for (int k = 0; k < ne; k++) {
            if (x[k] != 0) {
                if ((int64_t)out->residual_bits.size() == nres) break;
                bool bit;
                if (!rd.read_tail_bool(buf, len, &bit)) return FAIL();
                if (out->residual_bits.size() >= 480) return FAIL();   // heapless::Vec<bool,480> overflow
                out->residual_bits.push_back(bit);
            }
        }
    } else {
        for (int k = 0; k < si.lastnz; k += 2) {
            if (save_lev[k] > 0) {
                bool cont;
                if (!read_res_bit(x, rd, buf, len, k, &nres, &cont)) return FAIL();
                if (!cont) break;
                if (!read_res_bit(x, rd, buf, len, k + 1, &nres, &cont)) return FAIL();
                if (!cont) break;
            }
        }
    }

    // :140-145, wrapping i32 sum (release build) then & 0xFFFF
    uint32_t seed = 0;
    for (int k = 0; k < ne; k++) {
        uint32_t a = (uint32_t)(x[k] < 0 ? -x[k] : x[k]);
        seed += a * (uint32_t)k;
    }
    out->noise_filling_seed = (int32_t)seed & 0xFFFF;
    out->is_zero_frame = si.lastnz == 2 && x[0] == 0 && x[1] == 0 && si.global_gain_index == 0;
    out->frame_num_bits = nbits;
    return true;
}

// ================================================================== residual_spectrum.rs:13-39
void residual_spectrum_decode(bool lsb_mode, const uint8_t* bits, int nbits, float* spec, int ne) {
    if (lsb_mode) return;
    int i = 0;
    for (int k = 0; k < ne; k++) {
        if (spec[k] != 0.0f) {
            if (i >= nbits) break;
            if (bits[i++]) {
                if (spec[k] > 0.0f) spec[k] += 0.3125f; else spec[k] += 0.1875f;
            } else {
                if (spec[k] > 0.0f) spec[k] -= 0.1875f; else spec[k] -= 0.3125f;
            }
        }
    }
}

// ================================================================== noise_filling.rs:18-56
void apply_noise_filling(bool is_zero_frame, int32_t seed, int bandwidth, FrameDuration d, int noise_factor,
                         const int32_t* xi, float* xf, int ne) {
    if (is_zero_frame) return;
    static const int BW75[5] = {60, 120, 180, 240, 300}, BW10[5] = {80, 160, 240, 320, 400};
    int bw_stop = (d == SevenPointFiveMs ? BW75 : BW10)[bandwidth];
    int nf_start = d == SevenPointFiveMs ? 18 : 24, nf_width = d == SevenPointFiveMs ? 2 : 3;
    int32_t nf = seed;
    float level = (8.0f - (float)noise_factor) / 16.0f;
    int stop = bw_stop < ne ? bw_stop : ne;   // iter over spec_lines_float[..ne].take(bw_stop)
    for (int k = nf_start; k < stop; k++) {
        int from = k - nf_width;
        int to = (bw_stop - 1) < (k + nf_width) ? (bw_stop - 1) : (k + nf_width);
        bool all_zero = true;
        for (int j = from; j <= to; j++) if (xi[j] != 0) { all_zero = false; break; }
        if (all_zero) {
            nf = (13849 + nf * 31821) & 0xFFFF;
            xf[k] = nf < 0x8000 ? level : -level;
        }
    }
}

// ================================================================== global_gain.rs:15-25
void apply_global_gain(int frame_num_bits, int fs_ind, int gg_ind, float* spec, int ne) {
    int fs = fs_ind + 1;
    int q = frame_num_bits / (10 * fs);
    int gg_off = -(q < 115 ? q : 115) - 105 - (5 * fs);
    float exponent = ((float)gg_ind + (float)gg_off) / 28.0f;
    float gg = msun_powf(10.0f, exponent);
    for (int k = 0; k < ne; k++) spec[k] *= gg;
}

// ================================================================== temporal_noise_shaping.rs:24-138
void apply_tns_decode(FrameDuration d, int bandwidth, int num_tns_filters, const int* rc_order, const int* rc_i,
                      int n_rc_i, float* spec) {
    // band split :83-138
    int start[2], stop[2], nbands;
    if (d == TenMs) {
        static const int S1[3] = {80, 160, 240};
        if (bandwidth < 3) { nbands = 1; start[0] = 12; stop[0] = S1[bandwidth]; }
        else if (bandwidth == 3) { nbands = 2; start[0] = 12; stop[0] = 160; start[1] = 160; stop[1] = 320; }
        else { nbands = 2; start[0] = 12; stop[0] = 200; start[1] = 200; stop[1] = 400; }
    } else {
        static const int S1[3] = {60, 120, 180};
        if (bandwidth < 3) { nbands = 1; start[0] = 9; stop[0] = S1[bandwidth]; }
        else if (bandwidth == 3) { nbands = 2; start[0] = 9; stop[0] = 120; start[1] = 120; stop[1] = 240; }
        else { nbands = 2; start[0] = 9; stop[0] = 150; start[1] = 150; stop[1] = 300; }
    }
    float rc_q[16];
    for (int i = 0; i < 16; i++) rc_q[i] = 0.0f;
    const float step = (float)(M_PI / 17.0);
    // QUIRK: index 0 is skipped, leaving rc = 0.0 (spec: sin(-8*pi/17)).  zip() stops at the shorter slice.
    for (int i = 0; i < 16 && i < n_rc_i; i++)
        if (rc_i[i] != 0) rc_q[i] = msun_sinf(step * (float)(rc_i[i] - 8));
    float st[8] = {0, 0, 0, 0, 0, 0, 0, 0};   // QUIRK: not reset between filters
    int nf = nbands < num_tns_filters ? nbands : num_tns_filters;
    for (int f = 0; f < nf; f++) {
        int order = rc_order[f];
        if (order <= 0) continue;
        int off = f * 8;
        for (int n = start[f]; n < stop[f]; n++) {
            int k = order - 1;
            float t = spec[n] - rc_q[k + off] * st[k];
            for (k = order - 2; k >= 0; k--) {
                float rc = rc_q[k + off];
                t -= rc * st[k];
                st[k + 1] = rc * t + st[k];
            }
            spec[n] = t;
            st[0] = t;
        }
    }
}

// ================================================================== spectral_noise_shaping.rs
// :155-235
void mpvq_deenum(int dim_in, int k_val_in, int ls_ind, uint32_t mpvq_ind, int32_t* vec_out) {
    for (int i = 0; i < dim_in; i++) vec_out[i] = 0;
    int leading_sign = ls_ind == 0 ? 1 : -1;
    int k_max_local = k_val_in;
    uint32_t ind = mpvq_ind;
    for (int pos = 0; pos < dim_in; pos++) {
        const uint32_t* h_row = LC3T_MPVQ_OFFSETS[dim_in - 1 - pos];
        int k_delta;
        if (ind != 0) {
            int k_acc = k_max_local;
            uint32_t off = h_row[k_acc];
            bool wrap_flag = ind < off;
            uint32_t ul_diff = 0;
            if (!wrap_flag) ul_diff = ind - off;
            while (wrap_flag) {
                k_acc -= 1;
                wrap_flag = ind < h_row[k_acc];
                if (!wrap_flag) ul_diff = ind - h_row[k_acc];
            }
            ind = ul_diff;
            k_delta = k_max_local - k_acc;
        } else {
            vec_out[pos] = leading_sign < 0 ? -k_max_local : k_max_local;
            break;
        }
        if (k_delta != 0) {
            vec_out[pos] = leading_sign < 0 ? -k_delta : k_delta;
            leading_sign = (ind & 1) ? -1 : 1;
            ind >>= 1;
            k_max_local -= k_delta;
        }
    }
}

// :21-151
void sns_decode(const Config& c, const SnsVq& s, float* spec) {
    float st1[16];
    for (int i = 0; i < 8; i++) { st1[i] = LC3T_LFCB[s.ind_lf][i]; st1[8 + i] = LC3T_HFCB[s.ind_hf][i]; }
    int shape_j = (s.submode_msb << 1) + s.submode_lsb;
    int32_t y[16] = {0}, z[16] = {0};
    const float* gains;
    switch (shape_j) {
        case 0:
            mpvq_deenum(10, 10, s.ls_inda, (uint32_t)s.idx_a, y);
            mpvq_deenum(6, 1, s.ls_indb, (uint32_t)s.idx_b, z);
            for (int i = 0; i < 6; i++) y[10 + i] = z[i];
            gains = LC3T_SNS_VQ_REG_ADJ_GAINS;
            break;
        case 1:
            mpvq_deenum(10, 10, s.ls_inda, (uint32_t)s.idx_a, y);
            for (int i = 10; i < 16; i++) y[i] = 0;
            gains = LC3T_SNS_VQ_REG_LF_ADJ_GAINS;
            break;
        case 2: mpvq_deenum(16, 8, s.ls_inda, (uint32_t)s.idx_a, y); gains = LC3T_SNS_VQ_NEAR_ADJ_GAINS; break;
        default: mpvq_deenum(16, 6, s.ls_inda, (uint32_t)s.idx_a, y); gains = LC3T_SNS_VQ_FAR_ADJ_GAINS; break;
    }
    float sum = 0.0f;
    for (int i = 0; i < 16; i++) sum += (float)y[i] * (float)y[i];
    float y_norm = std::sqrt(sum);
    float g = gains[s.g_ind];
    if (y_norm != 0.0f) g /= y_norm;
    float scf[16];
    for (int n = 0; n < 16; n++) {
        float factor = 0.0f;
        for (int col = 0; col < 16; col++) factor += (float)y[col] * LC3T_D[n][col];
        scf[n] = st1[n] + g * factor;
    }
    float si[64];
    si[0] = scf[0];
    si[1] = scf[0];
    for (int n = 0; n <= 14; n++) {
        float fn = scf[n], d = scf[n + 1] - fn;
        si[4 * n + 2] = fn + (1.0f / 8.0f * d);
        si[4 * n + 3] = fn + (3.0f / 8.0f * d);
        si[4 * n + 4] = fn + (5.0f / 8.0f * d);
        si[4 * n + 5] = fn + (7.0f / 8.0f * d);
    }
    si[62] = scf[15] + 1.0f / 8.0f * (scf[15] - scf[14]);
    si[63] = scf[15] + 3.0f / 8.0f * (scf[15] - scf[14]);
    int nb = c.nb, n2 = 64 - nb;
    if (n2 != 0) {
        for (int i = 0; i < n2; i++) si[i] = (si[2 * i] + si[2 * i + 1]) / 2.0f;
        for (int i = n2; i < nb; i++) si[i] = si[i + n2];
    }
    const uint16_t* ifs = band_indices(c);
    for (int b = 0; b < nb; b++) {
        float gs = fastmath_exp2_raw(si[b]);       // QUIRK: approximation is normative
        for (int k = ifs[b]; k < ifs[b + 1]; k++) spec[k] *= gs;
    }
}

// ================================================================== packet_loss_concealment.rs
void Plc::save(const float* spec) {                              // :50-54
    num_lost_frames = 0;
    alpha = 1.0f;
    std::memcpy(last_good.data(), spec, sizeof(float) * ne);
}
LtpfInfo Plc::load_into(float* spec, int n) {                    // :63-85
    if (num_lost_frames >= 4) alpha *= (num_lost_frames < 8) ? 0.9f : 0.85f;
    num_lost_frames += 1;
    int m = n < ne ? n : ne;
    for (int k = 0; k < m; k++) {
        plc_seed = (16831 + plc_seed * 12821) & 0xFFFF;
        spec[k] = plc_seed < 0x8000 ? last_good[k] * alpha : last_good[k] * -alpha;
    }
    return LtpfInfo{false, false, 0};
}

// ================================================================== modified_dct.rs (decoder)
void DecMdct::init(const Config& c, int transform_) {            // :24-74
    cfg = c;
    transform = transform_;
    dct.init(c.nf);
    if (transform == TRANSFORM_ENGINE) eng.init(c);
    mem_ola_add.assign(c.nf - c.z, 0.0f);
    t_hat.assign(2 * c.nf, 0.0f);
}
void DecMdct::run(const float* spec, float* freq) {              // :76-151
    int nf = cfg.nf, ne = cfg.ne, z = cfg.z, half = nf / 2;
    for (int k = 0; k < ne; k++) freq[k] = spec[k];
    for (int k = ne; k < nf; k++) freq[k] = 0.0f;
    float* t = t_hat.data();
    if (transform == TRANSFORM_ENGINE) {
        // the engine's DCT-IV, unfold and window; its head / tail are t[z + n] and t[nf + z + n] below
        eng.dct_iv(freq);
        eng.unfold(freq, t + z, t + nf + z);
        for (int n = 0; n < nf - z; n++) freq[n] = mem_ola_add[n] + t[z + n];
        for (int n = 0; n < nf - z; n++) mem_ola_add[n] = t[nf + z + n];
        for (int n = 0; n < z; n++) freq[nf - z + n] = t[nf + n];
        return;
    }
    dct.run(freq);
    // apply_mdct_inverse :97-136: t = [y, -rev(y)] rotated left by nf/2, wrapped quarter negated
    for (int n = 0; n < nf; n++) t[n] = freq[n];
    for (int n = 0; n < nf; n++) t[nf + n] = -freq[nf - 1 - n];
    std::vector<float> scratch(t, t + half);
    for (int n = 0; n < half; n++) t[n] = t[half + n];
    for (int n = 0; n < half; n++) t[half + n] = t[nf + n];
    for (int n = 0; n < half; n++) t[nf + n] = t[nf + half + n];
    for (int n = 0; n < half; n++) t[3 * half + n] = -scratch[n];
    float gain = 1.0f / std::sqrt(2.0f * (float)nf);
    for (int n = 0; n < 2 * nf; n++) t[n] *= gain;
    const float* w = mdct_window(cfg);
    for (int n = 0; n < 2 * nf; n++) t[n] *= w[2 * nf - 1 - n];  // :89
    // overlap_add :138-151
    for (int n = 0; n < nf - z; n++) freq[n] = mem_ola_add[n] + t[z + n];
    for (int n = 0; n < nf - z; n++) mem_ola_add[n] = t[nf + z + n];
    for (int n = 0; n < z; n++) freq[nf - z + n] = t[nf + n];
}

// ================================================================== long_term_post_filter.rs (decoder)
void DecLtpf::init(const Config& c) {                            // :60-134
    cfg = c;
    switch (c.fs) {
        case 8000: case 16000: l_den = 4; break;
        case 24000: l_den = 6; break;
        case 32000: l_den = 8; break;
        case 44100: l_den = 11; break;       // QUIRK: 11, with the 48 kHz tables truncated by zip()
        default: l_den = 12; break;
    }
    l_num = l_den - 2;
    if (c.n_ms == TenMs) { num_mem_blocks = 2; norm = c.nf / 4; } else { num_mem_blocks = 3; norm = c.nf / 3; }
    x_hat_mem.assign(c.nf * num_mem_blocks, 0.0f);
    x_hat_ltpf_mem.assign(c.nf * num_mem_blocks, 0.0f);
    c_num.assign(l_num + 1, 0.0f);
    c_den.assign(l_den + 1, 0.0f);
    c_num_mem = c_num;
    c_den_mem = c_den;
    scratch.assign(l_num + norm, 0.0f);
    ltpf_active_prev = false;
    block_start_index = 0;
    p_int_mem = p_fr_mem = 0;
}
int DecLtpf::wrap(int idx) const { return idx < 0 ? idx + num_mem_blocks * cfg.nf : idx; }   // :244-250
float DecLtpf::filt(int start, int pitch_int, const std::vector<float>& cn, const std::vector<float>& cd) const {
    int lden = (int)c_den.size() - 1;                            // :380-415
    float out = 0.0f;
    for (size_t k = 0; k < cn.size(); k++) out += cn[k] * x_hat_mem[wrap(start - (int)k)];
    int sden = start - pitch_int + lden / 2;
    for (size_t k = 0; k < cd.size(); k++) out -= cd[k] * x_hat_ltpf_mem[wrap(sden - (int)k)];
    return out;
}
void DecLtpf::run(const LtpfInfo& info, int nbits, float* freq) {   // :252-343
    const int nf = cfg.nf;
    // compute_filter_parameters :164-190
    int pitch_int = 0, pitch_frac = 0;
    if (info.is_active) {
        int pi = info.pitch_index, p_i;
        double p_f;
        if (pi >= 440) { p_i = pi - 283; p_f = 0.0; }
        else if (pi >= 380) { p_i = pi / 2 - 63; p_f = (double)(2 * pi - 4 * p_i - 252); }
        else { p_i = pi / 4 + 32; p_f = (double)(pi + 128 - 4 * p_i); }
        double pitch = (double)p_i + p_f / 4.0;
        double pitch_fs = pitch * (8000.0 * std::ceil((double)cfg.fs / 8000.0) / 12800.0);
        int p_up = (int)rust_f64_to_usize((pitch_fs * 4.0) + 0.5);
        pitch_int = p_up / 4;
        pitch_frac = p_up - 4 * pitch_int;
    }
    // compute_filter_coeffs :192-242
    c_num_mem = c_num;
    c_den_mem = c_den;
    if (!info.is_active) {
        std::fill(c_num.begin(), c_num.end(), 0.0f);
        std::fill(c_den.begin(), c_den.end(), 0.0f);
    } else {
        // compute_gains_params :142-161
        int t_nbits = cfg.n_ms == SevenPointFiveMs ? (int)rust_f64_to_usize(std::round((double)nbits * 10.0 / 7.5))
                                                   : nbits;
        int sf = cfg.fs_ind * 80;
        float gain;
        int gain_ind;
        if (t_nbits < 320 + sf) { gain = 0.4f; gain_ind = 0; }
        else if (t_nbits < 400 + sf) { gain = 0.35f; gain_ind = 1; }
        else if (t_nbits < 480 + sf) { gain = 0.3f; gain_ind = 2; }
        else if (t_nbits < 560 + sf) { gain = 0.25f; gain_ind = 3; }
        else { gain = 0.0f; gain_ind = 0; }   // QUIRK: filter stays "active" with zero coefficients
        const float *tn, *td;
        int ln, ld;
        switch (cfg.fs) {
            case 8000: tn = LC3T_TAB_LTPF_NUM_8000[gain_ind]; td = LC3T_TAB_LTPF_DEN_8000[pitch_frac]; ln = 3; ld = 5; break;
            case 16000: tn = LC3T_TAB_LTPF_NUM_16000[gain_ind]; td = LC3T_TAB_LTPF_DEN_16000[pitch_frac]; ln = 3; ld = 5; break;
            case 24000: tn = LC3T_TAB_LTPF_NUM_24000[gain_ind]; td = LC3T_TAB_LTPF_DEN_24000[pitch_frac]; ln = 5; ld = 7; break;
            case 32000: tn = LC3T_TAB_LTPF_NUM_32000[gain_ind]; td = LC3T_TAB_LTPF_DEN_32000[pitch_frac]; ln = 7; ld = 9; break;
            default: tn = LC3T_TAB_LTPF_NUM_48000[gain_ind]; td = LC3T_TAB_LTPF_DEN_48000[pitch_frac]; ln = 11; ld = 13; break;
        }
        for (size_t k = 0; k < c_num.size() && (int)k < ln; k++) c_num[k] = 0.85f * gain * tn[k];
        for (size_t k = 0; k < c_den.size() && (int)k < ld; k++) c_den[k] = gain * td[k];
    }

    const int blk = block_start_index;
    for (int n = 0; n < nf; n++) x_hat_mem[blk + n] = freq[n];
    const int s2p5 = (cfg.fs == 44100) ? 48000 / 400 : cfg.fs / 400;
    float* y = x_hat_ltpf_mem.data();
    const float* x = x_hat_mem.data();
    const float fnorm = (float)norm;

    auto deactivate_first = [&]() {                              // :417-424
        for (int n = 0; n < s2p5; n++) {
            y[blk + n] = x[blk + n];
            float fo = filt(blk + n, p_int_mem, c_num_mem, c_den_mem);
            fo *= 1.0f - ((float)n / fnorm);
            y[blk + n] -= fo;
        }
    };

    if (!info.is_active && !ltpf_active_prev) {                  // case 1
        for (int n = 0; n < nf; n++) y[blk + n] = x[blk + n];
    } else if (info.is_active && !ltpf_active_prev) {            // case 2
        for (int n = 0; n < s2p5; n++) {
            y[blk + n] = x[blk + n];
            float fo = filt(blk + n, pitch_int, c_num, c_den);
            fo *= (float)n / fnorm;
            y[blk + n] -= fo;
        }
        for (int n = s2p5; n < nf; n++) {
            y[blk + n] = x[blk + n];
            y[blk + n] -= filt(blk + n, pitch_int, c_num, c_den);
        }
    } else if (!info.is_active && ltpf_active_prev) {            // case 3
        deactivate_first();
        for (int n = s2p5; n < nf; n++) y[blk + n] = x[blk + n];
    } else if (pitch_int == p_int_mem && pitch_frac == p_fr_mem) {   // case 4
        for (int n = 0; n < nf; n++) {
            y[blk + n] = x[blk + n];
            y[blk + n] -= filt(blk + n, pitch_int, c_num, c_den);
        }
    } else {                                                     // case 5
        deactivate_first();
        // activate_first_2p5ms_from_mem :345-378
        if (blk < l_num) {
            int from = num_mem_blocks * nf - l_num;
            for (int i = 0; i < l_num; i++) scratch[i] = y[from + i];
            for (int i = 0; i < norm; i++) scratch[l_num + i] = y[i];
        } else {
            for (int i = 0; i < l_num + norm; i++) scratch[i] = y[blk - l_num + i];
        }
        for (int n = 0; n < s2p5; n++) {
            y[blk + n] = scratch[n + l_num];
            int lden = (int)c_den.size() - 1;
            float fo = 0.0f;
            int sn = l_num + n;
            for (size_t k = 0; k < c_num.size(); k++) fo += c_num[k] * scratch[sn - (int)k];
            int sd = (blk + n) - pitch_int + lden / 2;
            for (size_t k = 0; k < c_den.size(); k++) fo -= c_den[k] * y[wrap(sd - (int)k)];
            fo *= (float)n / fnorm;
            y[blk + n] -= fo;
        }
        for (int n = s2p5; n < nf; n++) {
            y[blk + n] = x[blk + n];
            y[blk + n] -= filt(blk + n, pitch_int, c_num, c_den);
        }
    }
    for (int n = 0; n < nf; n++) freq[n] = y[blk + n];
    block_start_index += nf;
    if (block_start_index > (num_mem_blocks - 1) * nf) block_start_index = 0;
    ltpf_active_prev = info.is_active;
    p_int_mem = pitch_int;
    p_fr_mem = pitch_frac;
}

// ================================================================== output_scaling.rs:13-26
void scale_and_round(const float* x, int n, int16_t* out) {
    for (int i = 0; i < n; i++) {
        int32_t tmp = x[i] > 0.0f ? rust_f32_to_i32(x[i] + 0.5f) : rust_f32_to_i32(x[i] - 0.5f);
        if (tmp > 32767) tmp = 32767;
        if (tmp < -32768) tmp = -32768;
        out[i] = (int16_t)tmp;
    }
}

// ================================================================== lc3_decoder.rs
void DecoderChannel::init(SamplingFrequency sf, FrameDuration fd, int transform) {   // :181-215 (zeroed buffers)
    cfg = make_config(sf, fd);
    spec.assign(cfg.ne, 0.0f);
    freq.assign(cfg.nf, 0.0f);
    plc.init(cfg.ne);
    mdct.init(cfg, transform);
    ltpf.init(cfg);
    frame_index = 0;
}

int DecoderChannel::decode(int bits_per_sample, const uint8_t* buf, int64_t len, int16_t* out, int n_out) {   // :73-154
    if (bits_per_sample != 16) return 1;
    frame_index += 1;
    int nbits = (int)len * 8;
    std::memset(last_x, 0, sizeof(last_x));
    BufferReader rd;
    SideInfo si;
    ArithmeticData ad;
    LtpfInfo pf;
    bool ok = read_side_info(buf, len, rd, cfg.fs_ind, cfg.ne, &si) &&
              arithmetic_decode(buf, len, rd, cfg.fs_ind, cfg.ne, si, cfg.n_ms, last_x, &ad);
    last_ok = ok;
    if (ok) {
        last_si = si;
        last_ad = ad;
        for (int k = 0; k < cfg.ne; k++) spec[k] = (float)last_x[k];
        residual_spectrum_decode(si.lsb_mode, ad.residual_bits.data(), (int)ad.residual_bits.size(), spec.data(), cfg.ne);
        apply_noise_filling(ad.is_zero_frame, ad.noise_filling_seed, si.bandwidth, cfg.n_ms, si.noise_factor, last_x,
                            spec.data(), cfg.ne);
        apply_global_gain(ad.frame_num_bits, cfg.fs_ind, si.global_gain_index, spec.data(), cfg.ne);
        apply_tns_decode(cfg.n_ms, si.bandwidth, si.num_tns_filters, ad.rc_order, ad.rc_i, 16, spec.data());
        sns_decode(cfg, si.sns_vq, spec.data());
        plc.save(spec.data());
        pf = si.ltpf;
    } else {
        pf = plc.load_into(spec.data(), cfg.ne);                 // errors are swallowed :138-141
    }
    mdct.run(spec.data(), freq.data());
    ltpf.run(pf, nbits, freq.data());
    scale_and_round(freq.data(), n_out < cfg.nf ? n_out : cfg.nf, out);   // zip() truncates
    return 0;
}

}  // namespace lc3o
