// lc3b engine, encoder kernels 2-5 of 5: spectrum + analysis results -> bitstream, one WARP per frame.
// Four kernels (BW/SNS, TNS, quantise: gain search + rate loop, bitstream) so that each one's code stays near
// the SM's 32 KB L1.5 instruction cache: as ONE kernel the 14k-instruction body made instruction fetch the top stall
// (49 % of samples), every resident warp being in a different phase.
// Compiled with -fmad=false: every expression below rounds exactly like the reference's f32 code.
//
// Replaces, per stream, the second half of EncoderChannel::encode (src/encoder/lc3_encoder.rs:74-110):
//   BandwidthDetector::run          src/encoder/bandwidth_detector.rs:64
//   SpectralNoiseShaping::run       src/encoder/spectral_noise_shaping.rs:203 (two-stage VQ :318/:363, MPVQ enumeration :585)
//   TemporalNoiseShaping::run       src/encoder/temporal_noise_shaping.rs:40 (autocorrelation, Levinson-Durbin, lattice)
//   SpectralQuantization::run       src/encoder/spectral_quantization.rs:75 (gain bisection, bit consumption, adjustment)
//   ResidualBitsEncoder::encode     src/encoder/residual_spectrum.rs:33
//   NoiseLevelEstimation            src/encoder/noise_level_estimation.rs:21
//   BitstreamEncoding::encode       src/encoder/bitstream_encoding.rs:77 with BufferWriter (buffer_writer.rs:5)
//
// The frame lives in the warp's slice of shared memory.  The byte-identity bar fixes the ORDER of every f32 sum,
// so the work is split along the axes that leave each sum intact:
//   * independent results go to different lanes (64 band energies, 32 codebook rows, 27 autocorrelation sums,
//     100 four-line energies, 400 quantised lines, 200 two-tuples of the context walk);
//   * a long ordered sum keeps its order: its terms are produced in parallel and one chain adds them;
//   * the TNS analysis lattice is FIR: its stages run one after the other, each over all lines at once;
//   * integer accumulations (bit estimates, ranks, offsets) are exact in any order and use warp scans;
//   * the range coder consumes a queue of (cumulative, frequency) pairs the lanes prepared, and the backward
//     side-bit stream is assembled by the lanes at prefix-summed offsets.
// The reference writes both ends of the frame interleaved; when they never meet the result is the OR of the two
// streams, which is what the fast path builds.  A frame whose two ends collide (the encoder overspent its budget)
// is re-encoded by one lane with the reference's interleaved write order (bitstream_encode_serial).
#include <string.h>

#include "lc3b_enc_common.cuh"
#include "lc3b_plan.cuh"
#include "lc3b_math.cuh"
#include "lc3_tables.h"

namespace lc3b {

struct QuantParams {
    const EncConfig* cfg;
    int n_streams, nbytes;
    size_t frame_stride;
    float* xf;
    const float* e_b;
    const int32_t* ehand;
    int32_t* estate;
    int16_t* xq;
    int32_t* qhand;
    uint8_t* lsbs;
    uint32_t* bs_scratch;
    int bs_words;
    uint8_t* frames_out;
    int w_bytes, w_bytes_fin, side_words, sym_cap, out_words;     // per-warp shared-memory slices (prepare / finish kernels)
    int inline_ac;     // small batches: the finish kernel runs the range coder itself (all lanes, same chain) and C2 is skipped
    const int32_t* ids;   // subset call: row u's rate-loop state is that of handle stream ids[u] (enc_quantize_kernel<false, true>)
    const int32_t* rows;  // time-parallel call: the row table (lc3b_common.cuh), n_streams its rows (enc_quantize_kernel<true, true>)
};

constexpr int QW = 8;                       // frames (warps) per CTA
constexpr int QNT_THREADS = QW * 32;
constexpr unsigned FULL = 0xffffffffu;
constexpr int NE_MAX = 400;
constexpr int S_FLOATS = 384;               // per-warp scratch
constexpr int TAIL_WORDS = 26;              // 800 deferred LSB / 400 residual bits

struct BwRes { int bw, nbits; };
struct SnsRes { int ind_lf, ind_hf, shape_j, gind, ls_inda, ls_indb; uint64_t joint; };
struct TnsRes { int nbits_tns, lpc_weighting, num_filters; int rc_order[2]; const int* rc_i; };
struct QRes { int gg_ind, nbits_spec, nbits_lsb, nbits_trunc, lsb_mode, rate_flag, lastnz_trunc; float gg; };

// Constant tables live at namespace scope: a function-local 64-bit table (msun's exp2f) was observed to be laid
// over live stack data by nvcc 12.9 at -O3, so nothing table-like is left on the stack in this file.
__device__ const int START10[4][4] = {{53, 0, 0, 0}, {47, 59, 0, 0}, {44, 54, 60, 0}, {41, 51, 57, 61}};   // bandwidth_detector.rs:5-18
__device__ const int STOP10[4][4] = {{63, 0, 0, 0}, {56, 63, 0, 0}, {52, 59, 63, 0}, {49, 55, 60, 63}};
__device__ const int START75[4][4] = {{51, 0, 0, 0}, {45, 58, 0, 0}, {42, 53, 60, 0}, {40, 51, 57, 61}};
__device__ const int STOP75[4][4] = {{63, 0, 0, 0}, {55, 63, 0, 0}, {51, 58, 63, 0}, {48, 55, 60, 63}};
__device__ const int NBITS_BW[5] = {0, 1, 2, 2, 3};
__device__ const int QUIET[4] = {20, 10, 10, 10}, CUTOFF[4] = {15, 23, 20, 20};
__device__ const int L10[4] = {4, 4, 3, 1}, L75[4] = {4, 4, 3, 2};
__device__ const float SNS_W[6] = {1.0f / 12.0f, 2.0f / 12.0f, 3.0f / 12.0f, 3.0f / 12.0f, 2.0f / 12.0f, 1.0f / 12.0f};   // spectral_noise_shaping.rs:59
__device__ const float TNS_LAG[9] = {1.0f, 0.9980280260203829f, 0.9921354055113971f, 0.9823915844707989f, 0.9689107911912967f,
                                     0.9518498073692735f, 0.9314049334023056f, 0.9078082299969592f, 0.8813231366694713f};   // temporal_noise_shaping.rs:81-84
__device__ const int GGA_T1[5] = {80, 230, 380, 530, 680}, GGA_T2[5] = {500, 1025, 1550, 2075, 2600},
                     GGA_T3[5] = {850, 1700, 2550, 3400, 4250};   // spectral_quantization.rs:351-353

__device__ __forceinline__ float shf(float v, int src) { return __shfl_sync(FULL, v, src); }
__device__ __forceinline__ int shi(int v, int src) { return __shfl_sync(FULL, v, src); }

// Lexicographic (value, index) minimum over the warp: the result of the reference's `if d < d_min` scan over
// ascending indices.  NaN and +inf never win; *idx comes back as the smallest contributed index when nothing does.
__device__ __forceinline__ void warp_argmin(float& v, int& idx) {
    if (!(v < INFINITY)) v = INFINITY;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        const float ov = __shfl_xor_sync(FULL, v, off);
        const int oi = __shfl_xor_sync(FULL, idx, off);
        if (ov < v || (ov == v && oi < idx)) { v = ov; idx = oi; }
    }
}
__device__ __forceinline__ int warp_sum_i(int v) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(FULL, v, off);
    return v;
}
__device__ __forceinline__ int warp_max_i(int v) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v = max(v, __shfl_xor_sync(FULL, v, off));
    return v;
}
__device__ __forceinline__ uint32_t warp_incl_scan(uint32_t v, int lane) {
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const uint32_t o = __shfl_up_sync(FULL, v, off);
        if (lane >= off) v += o;
    }
    return v;
}

// ---------------------------------------------------------------- bandwidth_detector.rs:64-127 (every lane, same values)
__device__ BwRes bandwidth_detect(const EncConfig& c, const float* e_b) {
    const int n_bw = c.fs_ind, nbits = NBITS_BW[n_bw];
    if (n_bw == 0) return {0, nbits};
    const bool d10 = c.n_ms == LC3B_10MS;
    const int* start = (d10 ? START10 : START75)[n_bw - 1];
    const int* stop = (d10 ? STOP10 : STOP75)[n_bw - 1];
    const int* l = d10 ? L10 : L75;
    int bw = 0;
#pragma unroll 1
    for (int k = n_bw - 1; k >= 0; k--) {
        const float width = (float)(stop[k] + 1 - start[k]);
        float quiet = 0.0f;
#pragma unroll 1
        for (int n = start[k]; n <= stop[k]; n++) quiet += e_b[n] / width;
        if (quiet >= (float)QUIET[k]) { bw = k + 1; break; }
    }
    if (n_bw == bw) return {bw, nbits};
    float cutoff_max = 0.0f;
    const int l_bw = l[bw];
    const int from = start[bw] + 1 - l_bw, to = start[bw];
#pragma unroll 1
    for (int n = from; n < to; n++) {
        const float cutoff = e_b[n - l_bw] / e_b[n];
        cutoff_max = maxf_rs(cutoff, cutoff_max);
    }
    if (cutoff_max > (float)CUTOFF[bw]) return {bw, nbits};
    return {n_bw, nbits};
}

// ---------------------------------------------------------------- spectral_noise_shaping.rs
// add_unit_pulse :285-316 as one thread's work (inputs in shared memory).  The best-candidate scan keeps the reference's
// order (and its habit of leaving the LAST candidate's correlation/energy in the in-out arguments).  The scan is a serial
// chain, so the frames of a CTA run it side by side on the first lanes of warp 0 instead of each repeating it in 32 lanes.
__device__ __forceinline__ void add_unit_pulse_1(const float* ax, int* cand, int n_max, int k, int k_max, float& corr_xy, float& energy_y) {
    float corr_last = corr_xy, en_last = energy_y;
#pragma unroll 1
    for (int it = k; it < k_max; it++) {
        int n_best = 0;
        corr_xy = corr_last + ax[0];
        float best_corr_sq = corr_xy * corr_xy;
        float best_en = en_last + 2.0f * (float)cand[0] + 1.0f;
#pragma unroll 1
        for (int n_c = 1; n_c < n_max; n_c++) {
            corr_xy = corr_last + ax[n_c];
            energy_y = en_last + 2.0f * (float)cand[n_c] + 1.0f;
            if (corr_xy * corr_xy * best_en > best_corr_sq * energy_y) {
                n_best = n_c;
                best_corr_sq = corr_xy * corr_xy;
                best_en = energy_y;
            }
        }
        corr_last += ax[n_best];
        en_last += 2.0f * (float)cand[n_best] + 1.0f;
        cand[n_best] += 1;
    }
}

// normalize_candidate :629-648 (the squared norm is a sum of small integers: exact in any order)
__device__ __forceinline__ float normalize_w(int y, bool in_range) {
    const int yy = in_range ? y : 0;
    const int sq = warp_sum_i(yy * yy);
    const float norm = sqrtf((float)sq);
    float v = (float)yy;
    if (yy != 0) v /= norm;
    return v;
}

__device__ __noinline__ void mvpq_enum(uint64_t* index, int* lead_sign_ind, int dim_in, const int* vec_in) {   // :585-627
    int next_sign_ind = INT32_MIN;
    int8_t k_val_acc = 0;
    *index = 0;
    int n = 0;
    uint64_t tmp_h_row = LC3T_MPVQ_OFFSETS[n][0];
#pragma unroll 1
    for (int pos = dim_in - 1; pos >= 0; pos--) {
        const int8_t tmp_val = (int8_t)vec_in[pos];
        if (((uint32_t)next_sign_ind & 0x80000000u) == 0 && tmp_val != 0) *index = 2 * *index + (uint64_t)next_sign_ind;
        if (tmp_val < 0) next_sign_ind = 1;
        else if (tmp_val > 0) next_sign_ind = 0;
        *index += tmp_h_row;
        k_val_acc = (int8_t)(k_val_acc + (tmp_val < 0 ? -tmp_val : tmp_val));
        if (pos != 0) n += 1;
        tmp_h_row = (k_val_acc >= 11) ? LC3T_MPVQ_OFFSETS[n + 1][k_val_acc % 11] : LC3T_MPVQ_OFFSETS[n][k_val_acc];
    }
    *lead_sign_ind = next_sign_ind;
}

// sns_run_quant :318-582.  In: lane n < 16 holds scf[n].  Out: lane n < 16 holds scfq[n].
__device__ float sns_run_quant_w(float scf_v, float* S, SnsRes* res, int lane, int wib, int n_live) {
    float* xqs = S + 208;                 // [4][16] normalised shapes
    float* t2s = S + 192;                 // [16] rotated residual
    int* ys = (int*)(S + 320);            // [4][16] pulse vectors
    // exchange area of the pulse search (S + 272 .. 320): |t2rot| [16], pulse counts [16], corr / energy / first pulse
    const int n16 = lane & 15;
    // stage 1: lane i evaluates codebook row i of both halves
    float dlf = 0.0f, dhf = 0.0f;
#pragma unroll 1
    for (int n = 0; n < 8; n++) {
        const float a = shf(scf_v, n), b = shf(scf_v, 8 + n);
        dlf += (a - LC3T_LFCB[lane][n]) * (a - LC3T_LFCB[lane][n]);
        dhf += (b - LC3T_HFCB[lane][n]) * (b - LC3T_HFCB[lane][n]);
    }
    int ind_lf = lane, ind_hf = lane;
    warp_argmin(dlf, ind_lf);
    if (!(dlf < INFINITY)) ind_lf = 0;
    warp_argmin(dhf, ind_hf);
    if (!(dhf < INFINITY)) ind_hf = 0;
    const float st1 = n16 < 8 ? LC3T_LFCB[ind_lf][n16] : LC3T_HFCB[ind_hf][n16 - 8];
    const float r1 = scf_v - st1;
    // stage 2 target: t2rot = r1 * D
    float t2rot = 0.0f;
#pragma unroll 1
    for (int row = 0; row < 16; row++) t2rot += shf(r1, row) * LC3T_D[row][n16];
    const float ax = fabsf(t2rot);
    float abs_sum = 0.0f;
#pragma unroll 1
    for (int n = 0; n < 16; n++) abs_sum += shf(ax, n);
    const float proj = (6.0f - 1.0f) / abs_sum;
    int y3 = cast_i32(floorf(ax * proj));
    float corr_xy = 0.0f, energy_y = 0.0f;
    int k = 0;
#pragma unroll 1
    for (int n = 0; n < 16; n++) {
        const int yn = shi(y3, n);
        const float an = shf(ax, n);
        if (yn != 0) {
            k += yn;
            corr_xy += (float)yn * an;
            energy_y += (float)yn * (float)yn;
        }
    }
    // add_unit_pulse :285-316, run for all frames of the CTA by warp 0 (see add_unit_pulse_1)
    auto pulses = [&](int n_max, int k_from, int k_max, int& cand) {
        float* xa = S + 272;
        int* xc = (int*)(S + 288);
        float* sc = S + 304;
        __syncwarp();                                                    // the previous call's reads of the exchange area are done
        if (lane < 16) { xa[lane] = ax; xc[lane] = cand; }
        if (lane == 0) { sc[0] = corr_xy; sc[1] = energy_y; ((int*)sc)[2] = k_from; }
        asm volatile("bar.sync 1, %0;" ::"r"(n_live * 32) : "memory");
        if (wib == 0 && lane < n_live) {
            float* oS = S + (size_t)lane * (NE_MAX + S_FLOATS);         // warp `lane`'s scratch (this is warp 0)
            add_unit_pulse_1(oS + 272, (int*)(oS + 288), n_max, ((const int*)(oS + 304))[2], k_max, oS[304], oS[305]);
        }
        asm volatile("bar.sync 1, %0;" ::"r"(n_live * 32) : "memory");
        if (lane < 16) cand = xc[lane];
        corr_xy = sc[0];
        energy_y = sc[1];
    };
    pulses(16, k, 6, y3);
    int y2 = y3;
    pulses(16, 6, 8, y2);
    int y1 = lane < 10 ? y2 : 0;
    int k1 = 8;
#pragma unroll 1
    for (int n = 10; n < 16; n++) {
        const int yn = shi(y2, n);
        const float an = shf(ax, n);
        if (yn != 0) {
            k1 -= yn;
            corr_xy -= (float)yn * an;
            energy_y -= (float)yn * (float)yn;
        }
    }
    pulses(10, k1, 10, y1);
    int y0 = lane < 10 ? y1 : 0;
    {
        float max_abs_x = 0.0f;
        int n_best = 0;
#pragma unroll 1
        for (int n_c = 10; n_c < 16; n_c++) {
            const float an = shf(ax, n_c);
            if (an > max_abs_x) { max_abs_x = an; n_best = n_c; }
        }
        if (lane == n_best) y0 = 1;
    }
    if (t2rot < 0.0f) { y0 = -y0; y1 = -y1; y2 = -y2; y3 = -y3; }      // y1 is zero beyond n = 9 either way
    const bool lo16 = lane < 16;
    const float xq0 = normalize_w(y0, lo16), xq1 = normalize_w(y1, lane < 10), xq2 = normalize_w(y2, lo16),
                xq3 = normalize_w(y3, lo16);
    if (lo16) {
        xqs[lane] = xq0; xqs[16 + lane] = xq1; xqs[32 + lane] = xq2; xqs[48 + lane] = xq3;
        ys[lane] = y0; ys[16 + lane] = y1; ys[32 + lane] = y2; ys[48 + lane] = y3;
        t2s[lane] = t2rot;
    }
    __syncwarp();
    // shape / gain search: candidate c = lane, in the reference's (j, i) order
    int cj = 0, ci = 0;
    const float* gains = LC3T_SNS_VQ_REG_ADJ_GAINS;
    if (lane >= 7) { cj = 3; ci = lane - 7; gains = LC3T_SNS_VQ_FAR_ADJ_GAINS; }
    else if (lane >= 4) { cj = 2; ci = lane - 4; gains = LC3T_SNS_VQ_NEAR_ADJ_GAINS; }
    else if (lane >= 1) { cj = 1; ci = lane - 1; gains = LC3T_SNS_VQ_REG_LF_ADJ_GAINS; }
    float d = INFINITY, g_c = 0.0f;
    if (lane < 14) {
        g_c = gains[ci];
        d = 0.0f;
#pragma unroll 1
        for (int n = 0; n < 16; n++) {
            const float diff = t2s[n] - g_c * xqs[cj * 16 + n];
            d += diff * diff;
        }
    }
    int best = lane;
    warp_argmin(d, best);
    int shape_j = 0, gind = 0;
    float g_sel = 0.0f;
    if (d < INFINITY) {
        shape_j = best >= 7 ? 3 : best >= 4 ? 2 : best >= 1 ? 1 : 0;
        gind = best - (best >= 7 ? 7 : best >= 4 ? 4 : best >= 1 ? 1 : 0);
    }
    g_sel = d < INFINITY ? shf(g_c, best) : 0.0f;
    const int lsb_gain = gind & 1;
    uint64_t idxa = 0, idxb = 0;
    int ls_inda = 0, ls_indb = 0;
    uint64_t joint;
    switch (shape_j) {
        case 0:
            mvpq_enum(&idxa, &ls_inda, 10, ys);
            mvpq_enum(&idxb, &ls_indb, 6, ys + 10);
            joint = (2 * idxb + (uint64_t)(int64_t)ls_indb + 2) * 2390004ull + idxa;
            break;
        case 1:
            mvpq_enum(&idxa, &ls_inda, 10, ys + 16);
            joint = (uint64_t)lsb_gain * 2390004ull + idxa;
            break;
        case 2:
            mvpq_enum(&idxa, &ls_inda, 16, ys + 32);
            joint = idxa;
            break;
        default:
            mvpq_enum(&idxa, &ls_inda, 16, ys + 48);
            joint = 15158272ull + (uint64_t)lsb_gain + 2 * idxa;
            break;
    }
    float factor = 0.0f;
#pragma unroll 1
    for (int col = 0; col < 16; col++) factor += xqs[shape_j * 16 + col] * LC3T_D[n16][col];
    const float scfq = st1 + g_sel * factor;
    res->ind_lf = ind_lf; res->ind_hf = ind_hf; res->shape_j = shape_j; res->gind = gind;
    res->ls_inda = ls_inda; res->ls_indb = ls_indb; res->joint = joint;
    __syncwarp();
    return scfq;
}

// SpectralNoiseShaping::run :203-282.  S[0..64) holds the band energies on entry.
__device__ SnsRes sns_encode_w(const EncConfig& c, float* x, float* S, bool attack, int lane, int wib, int n_live) {
    const float* W = SNS_W;
    float* eb = S;
    float* e = S + 64;
    const int nb = c.nb, diff = 64 - nb;
    WARP_STRIDE_R(b, 64) {
        auto pad = [&](int j) -> float { return diff > 0 ? (j < 2 * diff ? eb[j >> 1] : eb[j - diff]) : eb[j]; };
        float v;
        if (b == 0) v = 0.75f * pad(0) + 0.25f * pad(1);
        else if (b == 63) v = 0.25f * pad(62) + 0.75f * pad(63);
        else v = 0.25f * pad(b - 1) + 0.5f * pad(b) + 0.25f * pad(b + 1);
        e[b] = v * c.pre_emph[b];
    }
    __syncwarp();
    float total = 0.0f;
#pragma unroll 1
    for (int b = 0; b < 64; b++) total += e[b];
    total = (total / 64.0f) * powi_nt(10.0f, -4);
    const float floor_ = maxf_rs(powi_nt(2.0f, -32), total);
    __syncwarp();
    WARP_STRIDE_R(b, 64) e[b] = log2f_msun(1.1920929e-07f + maxf_rs(e[b], floor_)) / 2.0f;
    __syncwarp();
    const int n16 = lane & 15;
    float ds;
    if (n16 == 0) {
        ds = W[0] * e[0];
#pragma unroll 1
        for (int k = 1; k < 6; k++) ds += W[k] * e[k - 1];
    } else if (n16 == 15) {
        ds = W[5] * e[63];
#pragma unroll 1
        for (int k = 0; k < 5; k++) ds += W[k] * e[60 + k - 1];
    } else {
        ds = 0.0f;
        const int from = 4 * n16 - 1;
#pragma unroll 1
        for (int k = 0; k < 6; k++) ds += W[k] * e[from + k];
    }
    float tot = 0.0f;
#pragma unroll 1
    for (int n = 0; n < 16; n++) tot += shf(ds, n);
    const float avg = tot / 16.0f;
    ds = 0.85f * (ds - avg);
    float scf = ds;
    if (attack) {
        const int lo = n16 - 2 < 0 ? 0 : n16 - 2, hi = n16 + 2 > 15 ? 15 : n16 + 2;
        float s = shf(ds, lo);
#pragma unroll 1
        for (int j = 1; j < 5; j++) {
            const float v = shf(ds, lo + j > 15 ? 15 : lo + j);
            if (lo + j <= hi) s += v;
        }
        scf = s / (float)(hi - lo + 1);
        float st = 0.0f;
#pragma unroll 1
        for (int n = 0; n < 16; n++) st += shf(scf, n);
        const float sa = st / 16.0f;
        const float att = c.n_ms == LC3B_10MS ? 0.5f : 0.3f;
        scf = att * (scf - sa);
    }
    SnsRes res;
    const float scfq = sns_run_quant_w(scf, S, &res, lane, wib, n_live);
    // 16 -> 64 interpolation :85-98 of the decoder's twin, then the nb < 64 folding and g = 2^-scf
    float* it = S + 64;
    float* gs = S;
    const float s00 = shf(scfq, 0);
#pragma unroll 1
    for (int j = 0; j < 2; j++) {
        const int b = lane + 32 * j;
        const int bb = b < 2 ? 2 : b;
        const int n = (bb - 2) >> 2, r = (bb - 2) & 3;
        const float cf = 0.125f + 0.25f * (float)r;
        const int i0 = n < 15 ? n : 15, i1 = n < 15 ? n + 1 : 14;
        const float s0 = shf(scfq, i0), s1 = shf(scfq, i1);
        float v = n < 15 ? s0 + (cf * (s1 - s0)) : s0 + (cf * (s0 - s1));
        if (b < 2) v = s00;
        it[b] = v;
    }
    __syncwarp();
    float itv[2];
#pragma unroll 1
    for (int j = 0; j < 2; j++) {
        const int b = lane + 32 * j;
        float v = it[b];
        if (diff > 0) {
            if (b < diff) v = (it[2 * b] + it[2 * b + 1]) / 2.0f;
            else if (b < nb) v = it[diff + 1];
        }
        itv[j] = v;
    }
    __syncwarp();
#pragma unroll 1
    for (int j = 0; j < 2; j++) gs[lane + 32 * j] = exp2f_msun(-itv[j]);
    __syncwarp();
    WARP_STRIDE_R(k, c.ne) {
        const int b = c.band_of[k];
        if (b < nb) x[k] *= gs[b];
    }
    __syncwarp();
    return res;
}

// ---------------------------------------------------------------- temporal_noise_shaping.rs
__device__ int8_t tns_to_int(float x) {
    auto cast_i8 = [](float v) -> int8_t {
        if (v != v) return 0;
        if (v >= 127.0f) return 127;
        if (v <= -128.0f) return -128;
        return (int8_t)v;
    };
    if (x >= 0.0f) return cast_i8(x + 0.5f);
    return cast_i8(-(-x + 0.5f));
}

struct TnsP { int nf; int start[2], stop[2], ss[2][3], se[2][3]; };
__device__ const TnsP TNS_T10[5] = {
    {1, {12, 160}, {80, 0}, {{12, 34, 57}, {0, 0, 0}}, {{34, 57, 80}, {0, 0, 0}}},
    {1, {12, 160}, {160, 0}, {{12, 61, 110}, {0, 0, 0}}, {{61, 110, 160}, {0, 0, 0}}},
    {1, {12, 160}, {200, 0}, {{12, 88, 164}, {0, 0, 0}}, {{88, 164, 240}, {0, 0, 0}}},
    {2, {12, 160}, {160, 320}, {{12, 61, 110}, {160, 213, 266}}, {{61, 110, 160}, {213, 266, 320}}},
    {2, {12, 200}, {200, 400}, {{12, 74, 137}, {200, 266, 333}}, {{74, 137, 200}, {266, 333, 400}}},
};
__device__ const TnsP TNS_T75[5] = {
    {1, {9, 120}, {60, 0}, {{9, 26, 43}, {0, 0, 0}}, {{26, 43, 60}, {0, 0, 0}}},
    {1, {9, 120}, {120, 0}, {{9, 46, 83}, {0, 0, 0}}, {{46, 83, 120}, {0, 0, 0}}},
    {1, {9, 120}, {180, 0}, {{9, 66, 123}, {0, 0, 0}}, {{66, 123, 180}, {0, 0, 0}}},
    {2, {9, 120}, {120, 240}, {{9, 46, 82}, {120, 159, 200}}, {{46, 82, 120}, {159, 200, 240}}},
    {2, {9, 150}, {150, 300}, {{9, 56, 103}, {150, 200, 250}}, {{56, 103, 150}, {200, 250, 300}}},
};

// An IEEE division is ~15 instructions inline; in straight-line register code that runs once per frame (Levinson-Durbin
// below is unrolled over register arrays) a call is cheaper than the instruction fetch of 60 inlined copies.
__device__ __noinline__ float fdiv_call(float a, float b) { return a / b; }

// TemporalNoiseShaping::run :40-78.  Scratch: ac[2][27] at S, raw reflection coefficients at S+64,
// results rc_i (int[16]) at S+256 and rc_q (float[16]) at S+272 (kept until the bitstream is written).
__device__ void tns_encode_w(const EncConfig& c, float* x, float* S, int p_bw, int nbits, bool near_nyquist, TnsRes& r, int lane) {
    const TnsP& tp = (c.n_ms == LC3B_10MS ? TNS_T10 : TNS_T75)[p_bw];
    float* ac = S;
    float* rc_raw = S + 64;
    int* rc_i = (int*)(S + 256);
    float* rc_q = S + 272;
    r.rc_i = rc_i;
    r.num_filters = tp.nf;
    r.lpc_weighting = (c.n_ms == LC3B_10MS ? nbits < 480 : nbits < 360) ? 1 : 0;
    const float* LAG = TNS_LAG;
    // compute_normalized_autocorrelation :80-115: 3 sub-blocks x 9 lags = 27 ordered sums per filter, one per lane
    for (int f = 0; f < tp.nf; f++) {
        if (lane < 27) {
            const int sb = lane / 9, lag = lane - 9 * sb;
            const int start = tp.ss[f][sb], stop = tp.se[f][sb];
            float acc = 0.0f;
            for (int n = start + lag; n < stop; n++) acc += x[n - lag] * x[n];
            ac[f * 27 + lane] = acc;
        }
    }
    __syncwarp();
    // the 27 quotients ac[sb][k] / ac[sb][0] of a filter are independent: one per lane instead of 27 divisions in a row on
    // every lane (the sums below still add them in the reference's order)
    float* qv = S + 128;                                    // [2][27]
    for (int f = 0; f < tp.nf; f++) {
        if (lane < 27) qv[f * 27 + lane] = ac[f * 27 + lane] / ac[f * 27 + (lane / 9) * 9];
    }
    __syncwarp();
    {   // Levinson-Durbin :204-232 and LPC weighting / LPC -> RC :234-257: lane f works on filter f
        const int f = (lane & 1) < tp.nf ? (lane & 1) : 0;
        const float* acf = ac + f * 27;
        const float* qf = qv + f * 27;
        float rr[9];
#pragma unroll
        for (int k = 0; k < 9; k++) {
            const float r0 = k == 0 ? 3.0f : 0.0f;
            float rk = 0.0f, e_prod = 1.0f;
#pragma unroll
            for (int sb = 0; sb < 3; sb++) {
                e_prod *= acf[sb * 9];
                rk += qf[sb * 9 + k];
            }
            rr[k] = (e_prod == 0.0f ? r0 : rk) * LAG[k];
        }
        float a[9], al[9];
#pragma unroll
        for (int i = 0; i < 9; i++) a[i] = al[i] = 0.0f;
        float e = rr[0];
        a[0] = 1.0f;
#pragma unroll
        for (int k = 1; k < 9; k++) {
#pragma unroll
            for (int i = 0; i < 9; i++) al[i] = a[i];
            float rc = 0.0f;
#pragma unroll
            for (int n = 0; n < k; n++) rc -= al[n] * rr[k - n];
            if (e != 0.0f) rc = fdiv_call(rc, e);
            a[0] = 1.0f;
#pragma unroll
            for (int n = 1; n < k; n++) a[n] = al[n] + rc * al[k - n];
            a[k] = rc;
            e *= 1.0f - rc * rc;
        }
        const float pred_gain = e == 0.0f ? rr[0] : rr[0] / e;
        float rcq[8];
        if (pred_gain > 1.5f && !near_nyquist) {
            float gamma = 1.0f;
            if (r.lpc_weighting > 0 && pred_gain < 2.0f) gamma -= (1.0f - 0.85f) * (2.0f - pred_gain) / (2.0f - 1.5f);
#pragma unroll
            for (int k = 0; k < 9; k++) a[k] *= powi_nt(gamma, k);
#pragma unroll
            for (int k = 8; k >= 1; k--) {
                rcq[k - 1] = a[k];
                const float ee = 1.0f - rcq[k - 1] * rcq[k - 1];
#pragma unroll
                for (int n = 1; n < k; n++) {
                    float v = a[n] - rcq[k - 1] * a[k - n];
                    v = fdiv_call(v, ee);
                    al[n] = v;
                }
#pragma unroll
                for (int n = 1; n < k; n++) a[n] = al[n];
            }
        } else {
#pragma unroll
            for (int k = 0; k < 8; k++) rcq[k] = 0.0f;
        }
        if (lane < tp.nf) {
#pragma unroll
            for (int k = 0; k < 8; k++) rc_raw[lane * 8 + k] = rcq[k];
        }
    }
    __syncwarp();
    if (lane < 16) {                                         // quantisation :259-283: one coefficient per lane
        const float step = (float)M_PI / 17.0f;
        int qi = 8;
        float qv = 0.0f;
        if (lane < 8 * tp.nf) {
            qi = (int)(tns_to_int(asinf_msun(rc_raw[lane]) / step) + 8);
            qv = c.tns_sin[qi];                              // sin(step * (rc_i - 8)), tabulated (17 arguments)
        }
        rc_i[lane] = qi;
        rc_q[lane] = qv;
    }
    __syncwarp();
    int nbits_tns = 0;
    for (int f = 0; f < 2; f++) {
        int k = 7;
        while (k >= 0 && rc_i[f * 8 + k] == 8) k--;
        r.rc_order[f] = f < tp.nf ? k + 1 : 0;
    }
    for (int f = 0; f < tp.nf; f++) {
        const int ob = r.rc_order[f] != 0 ? LC3T_AC_TNS_ORDER_BITS[r.lpc_weighting][r.rc_order[f] - 1] : 0;
        int cb = 0;
        for (int k = 0; k < r.rc_order[f]; k++) cb += LC3T_AC_TNS_COEF_BITS[k][rc_i[f * 8 + k]];
        nbits_tns += (int)ceilf((2048.0f + (float)ob + (float)cb) / 2048.0f);
    }
    r.nbits_tns = nbits_tns;
    // forward lattice :313-341.  It is an FIR lattice: with f_0[n] = b_0[n] = x[n],
    //   f_{k+1}[n] = f_k[n] + rc_k * b_k[n-1],   b_{k+1}[n] = rc_k * f_k[n] + b_k[n-1]     (st[k] is b_k[n-1])
    // stage k+1 of every line only needs stage k of lines n and n-1, so the recursion over lines that the reference
    // writes is not a dependence: the stages run one after the other, each over all lines at once, with exactly the
    // reference's operations per line and stage.  A lane owns C consecutive lines (C odd: conflict-free shared-memory
    // columns) in registers; b_k[n-1] of its first line comes from its neighbour, of the filter's first line from the
    // state, which survives from filter 0 to filter 1 (b_k of filter 0's last line).
    float st8[8] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
    for (int f = 0; f < tp.nf; f++) {
        const int order = r.rc_order[f];
        if (order == 0) continue;
        const int start = tp.start[f], N = tp.stop[f] - start;
        constexpr int CM = 13;                                     // ceil(388 / 32)
        const int C = ((N + 31) >> 5) | 1;
        const int n0 = lane * C;
        float F[CM], B[CM];
#pragma unroll
        for (int i = 0; i < CM; i++) {
            const int n = n0 + i;
            F[i] = B[i] = (i < C && n < N) ? x[start + n] : 0.0f;
        }
        const int last_lane = (N - 1) / C, last_i = (N - 1) - last_lane * C;
        __syncwarp();
#pragma unroll 1                                                   // a rolled loop stays in the instruction cache
        for (int k = 0; k < order; k++) {
            const float rq = rc_q[f * 8 + k];
            float b_last = 0.0f, b_end = 0.0f;                     // this lane's b_k of its last line / of line N-1
#pragma unroll
            for (int i = 0; i < CM; i++) {
                if (i == C - 1) b_last = B[i];
                if (i == last_i) b_end = B[i];
            }
            float up = __shfl_up_sync(FULL, b_last, 1);
            if (lane == 0) up = st8[k];
            st8[k] = __shfl_sync(FULL, b_end, last_lane);          // state left behind: b_k of the filter's last line
#pragma unroll
            for (int i = CM - 1; i >= 0; i--) {
                const float prev = i == 0 ? up : B[i - 1];         // b_k[n-1]
                const float fk = F[i];
                B[i] = rq * fk + prev;
                F[i] = fk + rq * prev;
            }
        }
#pragma unroll
        for (int i = 0; i < CM; i++) {
            const int n = n0 + i;
            if (i < C && n < N) x[start + n] = F[i];
        }
        __syncwarp();
    }
}

// ---------------------------------------------------------------- spectral_quantization.rs
struct BitCons { int rate_flag, lastnz, nbits_lsb, lastnz_trunc, nbits_est, nbits_trunc; bool mode_flag; };

// magnitude pair of a two-tuple after its escape levels, and the context digit it leaves behind (:333-346)
struct Tup { int q0, q1; uint32_t a0, b0, a, b; int L; };
__device__ __forceinline__ Tup tup_of(uint32_t w) {
    Tup t;
    t.q0 = (int)(int16_t)(w & 0xffffu);
    t.q1 = (int)(int16_t)(w >> 16);
    t.a0 = (uint32_t)(t.q0 < 0 ? -t.q0 : t.q0) & 0xffffu;
    t.b0 = (uint32_t)(t.q1 < 0 ? -t.q1 : t.q1) & 0xffffu;
    const uint32_t m = t.a0 > t.b0 ? t.a0 : t.b0;
    t.L = m < 4 ? 0 : 30 - __clz(m);                     // escapes: while max(a, b) >= 4 { a >>= 1; b >>= 1 }
    t.a = t.a0 >> t.L;
    t.b = t.b0 >> t.L;
    return t;
}
// bit i of x -> bit 2i (x < 2^16)
__device__ __forceinline__ uint32_t spread_bits(uint32_t x) {
    x = (x | (x << 8)) & 0x00ff00ffu;
    x = (x | (x << 4)) & 0x0f0f0f0fu;
    x = (x | (x << 2)) & 0x33333333u;
    x = (x | (x << 1)) & 0x55555555u;
    return x;
}
__device__ __forceinline__ int tup_digit(const Tup& t) {
    const int l = t.L < 3 ? t.L : 3;
    return l <= 1 ? 1 + (int)(t.a + t.b) * (l + 1) : 12 + l;
}

// compute_bit_consumption :265-348.  The context of tuple n is 16 * digit(n-2) + digit(n-1), so every tuple's cost
// is known from its own and its two predecessors' magnitudes: lane l walks tuples [l*CH, (l+1)*CH), the running
// totals the truncation test needs are integer prefix sums.
__device__ BitCons compute_bit_consumption_w(int ne, int fs_ind, const int16_t* xq, uint32_t* pre, int nbits, int nbits_spec, int lane) {
    BitCons bc;
    bc.rate_flag = nbits > (160 + fs_ind * 160) ? 512 : 0;
    bc.mode_flag = nbits >= (480 + fs_ind * 160);
    const uint32_t* xw = (const uint32_t*)xq;
    const int nt = ne >> 1;
    int last = -1;
    WARP_STRIDE(n, nt) if (xw[n] != 0) last = n;
    last = warp_max_i(last);
    const int lastnz = last < 0 ? 2 : 2 * last + 2;
    const int ntz = lastnz >> 1;
    const int CH = (ntz + 31) >> 5;                       // the tuples that exist, spread evenly over the lanes
    const int n0 = lane * CH;
    int d2 = 0, d1 = 0;                                   // digits of tuples n-2, n-1
    if (n0 >= 1 && n0 - 1 < ntz) d1 = tup_digit(tup_of(xw[n0 - 1]));
    if (n0 >= 2 && n0 - 2 < ntz) d2 = tup_digit(tup_of(xw[n0 - 2]));
    uint32_t est = 0;
    int lsb = 0;
    const int n1 = n0 + CH < ntz ? n0 + CH : ntz;
#pragma unroll 1
    for (int n = n0; n < n0 + CH; n++) if (n < n1) {
        const Tup t = tup_of(xw[n]);
        const int tc = d2 * 16 + d1 + bc.rate_flag + (2 * n > ne / 2 ? 256 : 0);
        // escape levels (:285-300): level lev uses the model of min(lev, 3), so levels 3.. all cost the same and the
        // walk over levels closes into four terms (integer arithmetic: any order) - no lane-dependent trip count
        const int L = t.L;
        const int pk0 = LC3T_AC_SPEC_LOOKUP[tc], pk1 = LC3T_AC_SPEC_LOOKUP[tc + 1024];
        const int pk2 = LC3T_AC_SPEC_LOOKUP[tc + 2048], pk3 = LC3T_AC_SPEC_LOOKUP[tc + 3072];
        const uint32_t e0 = LC3T_AC_SPEC_BITS[pk0][16], e1 = LC3T_AC_SPEC_BITS[pk1][16] + 2 * 2048;
        const uint32_t e2 = LC3T_AC_SPEC_BITS[pk2][16] + 2 * 2048, e3 = LC3T_AC_SPEC_BITS[pk3][16] + 2 * 2048;
        est += (L > 0 ? e0 : 0u) + (L > 1 ? e1 : 0u) + (L > 2 ? e2 : 0u) + (L > 3 ? (uint32_t)(L - 3) * e3 : 0u);
        if (L > 0) { if (bc.mode_flag) lsb += 2; else est += 2 * 2048; }
        const int pki = L == 0 ? pk0 : L == 1 ? pk1 : L == 2 ? pk2 : pk3;
        est += LC3T_AC_SPEC_BITS[pki][t.a + 4 * t.b];
        if (t.a0 > 0) est += 2048;
        if (t.b0 > 0) est += 2048;
        if (t.L > 0 && bc.mode_flag) {
            if ((t.a0 >> 1) == 0 && t.q0 != 0) lsb += 1;
            if ((t.b0 >> 1) == 0 && t.q1 != 0) lsb += 1;
        }
        pre[n] = est | ((t.q0 != 0 || t.q1 != 0) ? 0x80000000u : 0u);     // est < 2^31
        d2 = d1;
        d1 = tup_digit(t);
    }
    const uint32_t incl = warp_incl_scan(est, lane);
    const uint32_t base = incl - est;
    const uint32_t est_total = __shfl_sync(FULL, incl, 31);
    int qual = -1;                                        // last tuple of this lane that is non-zero and still fits
    uint32_t qual_est = 0;
#pragma unroll 1
    for (int n = n0; n < n0 + CH; n++) if (n < n1) {
        const uint32_t pv = pre[n];
        const uint32_t e_n = base + (pv & 0x7fffffffu);
        if ((pv >> 31) != 0 && (int)ceilf((float)e_n / 2048.0f) <= nbits_spec) { qual = n; qual_est = e_n; }
    }
    const int qmax = warp_max_i(qual);
    uint32_t trunc = 0;
    int lastnz_trunc = 2;
    if (qmax >= 0) {
        lastnz_trunc = 2 * qmax + 2;
        trunc = __shfl_sync(FULL, qual_est, qmax / CH);
    }
    bc.nbits_lsb = warp_sum_i(lsb);
    bc.lastnz = lastnz;
    bc.lastnz_trunc = lastnz_trunc;
    bc.nbits_est = (int)ceilf((float)est_total / 2048.0f) + bc.nbits_lsb;
    bc.nbits_trunc = (int)ceilf((float)trunc / 2048.0f);
    return bc;
}

__device__ float gain_of(const EncConfig& c, int gg_ind, int gg_off) {   // 10^((gg_ind + gg_off) / 28), :239
    const int idx = gg_ind + gg_off + 245;
    if (idx >= 0 && idx < 400) return c.gg_table[idx];
    return powf_msun(10.0f, ((float)gg_ind + (float)gg_off) / 28.0f);
}

__device__ __noinline__ BitCons quantize_spectrum_w(const EncConfig& c, const float* xf, int16_t* xq, uint32_t* pre, int nbits, int gg_off, int gg_ind,
                                       int nbits_spec, float* gg_out, bool* lsb_mode, int lane) {   // :230-263
    const int ne = c.ne;
    const float gg = gain_of(c, gg_ind, gg_off);
    WARP_STRIDE(k, ne) {
        const float v = xf[k];
        const float q = v / gg;                      // one division for both signs (the lanes of a warp mix them)
        xq[k] = cast_i16(v >= 0.0f ? q + 0.375f : q - 0.375f);
    }
    __syncwarp();
    BitCons bc = compute_bit_consumption_w(ne, c.fs_ind, xq, pre, nbits, nbits_spec, lane);
    __syncwarp();
    WARP_STRIDE_FROM(k, bc.lastnz_trunc, bc.lastnz) xq[k] = 0;
    __syncwarp();
    *gg_out = gg;
    *lsb_mode = bc.mode_flag && bc.nbits_est > nbits_spec;
    return bc;
}

// SpectralQuantization::run :75-120.  e4: [ne/4] energies, T: [224] scratch (bisection terms, then per-tuple bit prefixes).
constexpr size_t QUANTIZE_WARP_BYTES = sizeof(float) * (NE_MAX + 100 + 224) + sizeof(int16_t) * NE_MAX;   // xf | e4 | T | xq
__device__ QRes spectral_quantization_w(const EncConfig& c, int32_t* es, const float* xf, int16_t* xq, float* e4, float* T,
                                        int nbits, int nbits_bw, int nbits_tns, int nbits_ltpf, int lane, int wib, int n_live,
                                        uint8_t* smem_base) {
    const int ne = c.ne, fs_ind = c.fs_ind;
    int lg = 0;
    while ((1 << lg) < ne / 2) lg++;
    const int nbits_ari = lg + (nbits <= 1280 ? 3 : nbits <= 2560 ? 4 : 5);
    const int nbits_spec = nbits - (nbits_bw + nbits_tns + nbits_ltpf + 38 + 8 + 3 + nbits_ari);
    const bool reset_offset_old = es[ES_Q_RESET_OFFSET_OLD] != 0;
    const float nbits_offset_old = __uint_as_float((uint32_t)es[ES_Q_NBITS_OFFSET_OLD]);
    const int nbits_est_old = es[ES_Q_NBITS_EST_OLD];
    __syncwarp();                                                      // every lane has read the state before lane 0 updates it
    float nbits_offset;
    if (reset_offset_old) nbits_offset = 0.0f;
    else {
        const float prev = nbits_offset_old + (float)0 - (float)nbits_est_old;   // nbits_spec_old is never updated (:59)
        nbits_offset = 0.8f * nbits_offset_old + 0.2f * minf_rs(40.0f, maxf_rs(-40.0f, prev));
    }
    int nbits_spec_adj;
    {
        const float v = (float)nbits_spec + nbits_offset + 0.5f;       // `as u16`: saturating
        nbits_spec_adj = v != v ? 0 : v >= 65535.0f ? 65535 : v <= 0.0f ? 0 : (int)v;
    }
    const int q = (int16_t)nbits / (int16_t)(10 * (fs_ind + 1));
    const int gg_off = -(115 < q ? 115 : q) - 105 - 5 * (fs_ind + 1);
    const int ne4 = ne / 4;
    float xmax = 0.0f;                                                 // global_gain_limitation :212-228 (max is order-free)
    WARP_STRIDE(i, ne4) {                             // compute_spectral_energy :390-395
        const float4 p4 = ((const float4*)xf)[i];
        const float total = p4.x * p4.x + p4.y * p4.y + p4.z * p4.z + p4.w * p4.w;
        e4[i] = 10.0f * log10f_msun(1.1920929e-07f + total);
        xmax = maxf_rs(xmax, fabsf(p4.x));
        xmax = maxf_rs(xmax, fabsf(p4.y));
        xmax = maxf_rs(xmax, fabsf(p4.z));
        xmax = maxf_rs(xmax, fabsf(p4.w));
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) xmax = maxf_rs(xmax, __shfl_xor_sync(FULL, xmax, off));
    __syncwarp();
    // global_gain_estimation :174-210.  Per step: the 100 terms of the ordered sum are produced by the lanes (the
    // only coupling is "has a louder block been seen above me", a ballot), then added from the top down by one chain.
    int fac = 256, gg_ind = 255;
    const int rounds = (ne4 + 31) >> 5;
    // the block energies do not change over the eight bisection steps: their scaled forms (two f32 multiplications and
    // two IEEE divisions per block, exactly the reference's expressions) are computed once, not once per step
    float e28[4], e28x2[4], e28lo[4];
#pragma unroll
    for (int r = 0; r < 4; r++) {
        const int i = r * 32 + lane;
        const float ei = (r < rounds && i < ne4) ? e4[i] : -INFINITY;
        e28[r] = ei * 28.0f / 20.0f;
        e28lo[r] = ei * 28.0f / 20.0f - 43.0f * 28.0f / 20.0f;
        e28x2[r] = 2.0f * ei * 28.0f / 20.0f;
    }
    for (int it = 0; it < 8; it++) {
        fac >>= 1;
        gg_ind -= fac;
        const float g = (float)gg_ind + (float)gg_off;
        uint32_t ball[4];
#pragma unroll
        for (int r = 0; r < 4; r++) {
            const int i = r * 32 + lane;
            const bool loud = (r < rounds && i < ne4) && !(e28[r] < g);
            ball[r] = __ballot_sync(FULL, loud);
        }
        bool any_loud = false;
#pragma unroll
        for (int r = 3; r >= 0; r--) {
            const int i = r * 32 + lane;
            if (r < rounds && i < ne4) {
                const bool above = any_loud || (lane < 31 && (ball[r] >> (lane + 1)) != 0);
                float term;
                if (e28[r] < g) term = above ? 2.7f * 28.0f / 20.0f : 0.0f;
                else if (g < e28lo[r]) term = e28x2[r] - 2.0f * g - 36.0f * 28.0f / 20.0f;
                else term = e28[r] - g + 7.0f * 28.0f / 20.0f;
                T[i] = term;
            }
            any_loud = any_loud || ball[r] != 0;
        }
        const bool is_zero = !any_loud;
        // the ordered sum is one chain per frame: the chains of the CTA's frames run side by side on the first lanes of
        // warp 0 (between two named barriers) instead of each being repeated by the 32 lanes of its own warp
        asm volatile("bar.sync 1, %0;" ::"r"(n_live * 32) : "memory");
        if (wib == 0 && lane < n_live) {
            float* oT = (float*)(smem_base + (size_t)lane * QUANTIZE_WARP_BYTES) + NE_MAX + 100;   // warp `lane`'s T
            float acc = 0.0f;
            for (int i = ne4 - 1; i >= (ne4 & ~3); i--) acc += oT[i];
            for (int i4 = ne4 / 4 - 1; i4 >= 0; i4--) {
                const float4 t4 = ((const float4*)oT)[i4];
                acc += t4.w; acc += t4.z; acc += t4.y; acc += t4.x;
            }
            oT[208] = acc;
        }
        asm volatile("bar.sync 1, %0;" ::"r"(n_live * 32) : "memory");
        const float tmp = T[208];
        if ((tmp > (float)nbits_spec_adj * 1.4f * 28.0f / 20.0f) && !is_zero) gg_ind += fac;
    }
    int gg_min = 0;
    if (xmax > 0.0f) gg_min = (int)(int16_t)(cast_i16(ceilf(28.0f * log10f_msun(xmax / (32768.0f - 0.375f)))) - (int16_t)gg_off);
    bool reset_offset;
    if (gg_ind < gg_min || xmax == 0.0f) { reset_offset = true; gg_ind = gg_min; } else reset_offset = false;

    float gg;
    bool lsb_mode;
    BitCons bc = quantize_spectrum_w(c, xf, xq, (uint32_t*)T, nbits, gg_off, gg_ind, nbits_spec, &gg, &lsb_mode, lane);
    if (lane == 0) {
        es[ES_Q_NBITS_OFFSET_OLD] = (int32_t)__float_as_uint(nbits_offset);   // state saved BEFORE the adjustment (:96-100)
        es[ES_Q_NBITS_EST_OLD] = bc.nbits_est;
        es[ES_Q_RESET_OFFSET_OLD] = reset_offset;
    }
    const int t1 = GGA_T1[fs_ind], t2 = GGA_T2[fs_ind], t3 = GGA_T3[fs_ind];
    const int nbits_est = bc.nbits_est;
    float delta;
    if (nbits_est < t1) delta = ((float)nbits_est + 48.0f) / 16.0f;
    else if (nbits_est < t2) {
        const float tmp1 = (float)t1 / 16.0f + 3.0f, tmp2 = (float)t2 / 48.0f;
        delta = ((float)nbits_est - (float)t1) * (tmp2 - tmp1) / ((float)t2 - (float)t1) + tmp1;
    } else if (nbits_est < t3) delta = (float)nbits_est / 48.0f;
    else delta = (float)t3 / 48.0f;
    delta = floorf(delta + 0.5f);
    const float delta2 = delta + 2.0f;
    const int origin = gg_ind;
    if ((gg_ind < 255 && nbits_est > nbits_spec) || (gg_ind > 0 && (float)nbits_est < ((float)nbits_spec - delta2))) {
        if ((float)nbits_est < ((float)nbits_spec - delta2)) gg_ind -= 1;
        else if (gg_ind == 254 || (float)nbits_est < ((float)nbits_spec + delta)) gg_ind += 1;
        else gg_ind += 2;
        gg_ind = gg_ind > gg_min ? gg_ind : gg_min;
    }
    if (origin != gg_ind) bc = quantize_spectrum_w(c, xf, xq, (uint32_t*)T, nbits, gg_off, gg_ind, nbits_spec, &gg, &lsb_mode, lane);
    QRes r;
    r.gg_ind = gg_ind; r.nbits_spec = nbits_spec; r.nbits_lsb = bc.nbits_lsb; r.lsb_mode = lsb_mode;
    r.nbits_trunc = bc.nbits_trunc; r.rate_flag = bc.rate_flag; r.lastnz_trunc = bc.lastnz_trunc; r.gg = gg;
    return r;
}

// ---------------------------------------------------------------- residual_spectrum.rs:33-62
// One bit per non-zero line in line order, at most mx (and 400): ranks come from ballots.  Bits land in tail[].
__device__ int residual_bits_w(int ne, const float* xf, const int16_t* xq, float gg, int mx, uint32_t* tail, int lane) {
    if (mx <= 0) return 0;
    const int lim = mx < 400 ? mx : 400;
    int base = 0;
    for (int k0 = 0; k0 < ne && base < lim; k0 += 32) {
        const int k = k0 + lane;
        const int v = k < ne ? xq[k] : 0;
        const uint32_t nz = __ballot_sync(FULL, v != 0);
        const int rank = base + __popc(nz & ((1u << lane) - 1u));
        if (v != 0 && rank < lim && xf[k] >= (float)v * gg) atomicOr(&tail[rank >> 5], 1u << (rank & 31));
        base += __popc(nz);
    }
    return base < lim ? base : lim;
}

// ---------------------------------------------------------------- noise_level_estimation.rs:21-55
// The qualifying lines' |x|/gg replace the spectrum in place (0 elsewhere), then one chain adds them in line order.
__device__ int noise_factor_w(const EncConfig& c, float* xf, const int16_t* xq, int bw_ind, float gg, int lane, int wib, int n_live,
                              size_t warp_bytes) {
    const bool d10 = c.n_ms == LC3B_10MS;
    const int bw_stop = d10 ? 80 * (bw_ind + 1) : 60 * (bw_ind + 1);
    const int nf_start = d10 ? 24 : 18, nf_width = d10 ? 3 : 2;
    const int nf_stop = c.ne < bw_stop ? c.ne : bw_stop;
    int count = 0;                                                // qualifying lines so far (warp-uniform)
    // nzm[r] = ballot of "xq[32 r + lane] != 0"; a line's window [k - w, hi] is then a bit range of at most 7 bits
    uint32_t nzm[13];
#pragma unroll
    for (int r = 0; r < 13; r++) {
        const int k = 32 * r + lane;
        nzm[r] = __ballot_sync(FULL, k < c.ne && xq[k] != 0);
    }
    // The qualifying lines' |x| / gg are packed in line order into the front of xf (a line's value lands at or below
    // its own index, and each round's reads are done before its writes), so the ordered sum only walks those.
#pragma unroll
    for (int r = 0; r < 13; r++) {
        const int k = 32 * r + lane;
        bool quiet = false;
        float val = 0.0f;
        if (k >= nf_start && k < nf_stop) {
            const int hi = bw_stop - 1 < k + nf_width ? bw_stop - 1 : k + nf_width;
            const int lo = k - nf_width;
            // 64-bit view of words r-1, r, r+1 around the lane: bits [lo, hi] relative to 32 (r - 1)
            const uint32_t wm = r > 0 ? nzm[r - 1] : 0u, w0 = nzm[r], wp = r < 12 ? nzm[r + 1] : 0u;
            const int rel = lo - 32 * (r - 1);                     // 32 - w + lane >= 29
            const uint64_t lo64 = (uint64_t)wm | ((uint64_t)w0 << 32);
            const uint64_t hi64 = (uint64_t)w0 | ((uint64_t)wp << 32);
            const uint32_t win = rel < 32 ? (uint32_t)(lo64 >> rel) : (uint32_t)(hi64 >> (rel - 32));
            quiet = (win & ((1u << (hi - lo + 1)) - 1u)) == 0;
            if (quiet) val = fabsf(xf[k]) / gg;
        }
        const uint32_t qm = __ballot_sync(FULL, quiet);
        __syncwarp();
        if (quiet) xf[count + __popc(qm & ((1u << lane) - 1u))] = val;
        count += __popc(qm);
    }
    // the ordered sum is one chain per frame: the CTA's chains run side by side on the first lanes of warp 0
    if (lane == 0) ((int*)xf)[NE_MAX - 1] = count;                   // count <= ne - 24, so the last slot is free
    asm volatile("bar.sync 1, %0;" ::"r"(n_live * 32) : "memory");
    if (wib == 0 && lane < n_live) {
        float* oxf = (float*)((uint8_t*)xf + (size_t)lane * warp_bytes);   // warp `lane`'s spectrum buffer (this is warp 0)
        const int n = ((const int*)oxf)[NE_MAX - 1];
        float acc = 0.0f;
        for (int i = 0; i < n; i++) acc += oxf[i];
        oxf[NE_MAX - 2] = acc;
    }
    asm volatile("bar.sync 1, %0;" ::"r"(n_live * 32) : "memory");
    const float sum = xf[NE_MAX - 2];
    const float level = count > 0 ? sum / (float)count : 0.0f;
    const float diff = 8.0f - 16.0f * level;
    if (diff >= 0.0f) {
        const int v = cast_i32(diff + 0.5f);
        return v < 7 ? v : 7;
    }
    return 0;
}

// ---------------------------------------------------------------- bitstream_encoding.rs + buffer_writer.rs
// Reference-order writer, used by one lane when the frame's two ends collide.
struct Writer {
    uint8_t* buf;
    int nbytes;
    int bp;
    int bp_side;
    uint32_t mask_side;
    __device__ __noinline__ void bool_backward(bool bit) {                 // buffer_writer.rs:27-40
        if (bp_side >= 0) {
            if (!bit) buf[bp_side] &= (uint8_t)~mask_side; else buf[bp_side] |= (uint8_t)mask_side;
        }
        if (mask_side == 0x80) { mask_side = 1; bp_side -= 1; } else mask_side <<= 1;
    }
    __device__ __noinline__ void uint_backward(uint64_t val, int nbits) {   // :19-25
#pragma unroll 1
        for (int i = 0; i < nbits; i++) { bool_backward((val & 1) != 0); val >>= 1; }
    }
    __device__ __noinline__ void uint_forward(uint32_t val, int nbits) {    // :42-53 (QUIRK: bp is not advanced)
        uint32_t mask = 0x80;
        if (bp >= nbytes) return;
#pragma unroll 1
        for (int i = 0; i < nbits; i++) {
            if (((val & 0xff) & mask) == 0) buf[bp] &= (uint8_t)~mask; else buf[bp] |= (uint8_t)mask;
            mask >>= 1;
        }
    }
    __device__ __forceinline__ void byte_forward(uint32_t v) { if (bp < nbytes) buf[bp] = (uint8_t)v; bp++; }
    __device__ __forceinline__ int nbits_side_written(int nbits) const { return nbits - (8 * bp_side + 8 - (31 - __clz(mask_side))); }
};
struct AcEnc { uint32_t low, range; int cache, carry, carry_count; };

template <class W>
__device__ __forceinline__ void ac_shift(AcEnc& st, W& w) {              // bitstream_encoding.rs:397-415
    if (st.low < 0x00ff0000u || st.carry == 1) {
        if (st.cache >= 0) w.byte_forward((uint32_t)((st.cache + st.carry) & 0xff));
        while (st.carry_count > 0) {
            w.byte_forward((uint32_t)((st.carry + 0xff) & 0xff));
            st.carry_count -= 1;
        }
        st.cache = (int)(st.low >> 16);
        st.carry = 0;
    } else {
        st.carry_count += 1;
    }
    st.low <<= 8;
    st.low &= 0x00ffffffu;
}
template <class W>
__device__ __forceinline__ void ac_encode(AcEnc& st, W& w, int cum, int freq) {   // :417-429
    const uint32_t r = st.range >> 10;
    st.low += r * (uint32_t)cum;
    if (st.low >> 24 != 0) st.carry = 1;
    st.low &= 0x00ffffffu;
    st.range = r * (uint32_t)freq;
    while (st.range < 0x10000u) {
        st.range <<= 8;
        ac_shift(st, w);
    }
}
__device__ __noinline__ void ac_encode_serial(AcEnc& st, Writer& w, int cum, int freq) { ac_encode(st, w, cum, freq); }
// ac_enc_finish :354-395 up to (not including) the final partial byte; returns the bit count of that byte
template <class W>
__device__ __forceinline__ int ac_finish(AcEnc& st, W& w) {
    int bits = 1;
    while ((st.range >> (24 - bits)) == 0) bits++;
    uint32_t mask = 0x00ffffffu >> bits;
    uint32_t val = st.low + mask;
    const uint32_t over1 = val >> 24;
    const uint32_t high = st.low + st.range;
    const uint32_t over2 = high >> 24;
    val &= 0x00ffffffu & ~mask;
    if (over1 == over2) {
        if ((val + mask) >= high) {
            bits += 1;
            mask >>= 1;
            val = ((st.low + mask) & 0x00ffffffu) & ~mask;
        }
        if (val < st.low) st.carry = 1;
    }
    st.low = val;
    while (bits > 0) { ac_shift(st, w); bits -= 8; }
    bits += 8;
    return bits;
}

struct SideHdr {
    const BwRes* bw; const SnsRes* sns; const TnsRes* tns; const QRes* q;
    int pitch_present, ltpf_active, pitch_index, nf_factor, lg;
};

// side information in the reference's order (bitstream_encoding.rs:138-232) through any `put(value, nbits)`
template <class P>
__device__ __forceinline__ void write_side_info(const SideHdr& h, P& put) {
    if (h.bw->nbits > 0) put((uint64_t)h.bw->bw, h.bw->nbits);
    put((uint64_t)((h.q->lastnz_trunc >> 1) - 1), h.lg);
    put((uint64_t)(h.q->lsb_mode != 0), 1);
    put((uint64_t)(int64_t)h.q->gg_ind, 8);
    for (int f = 0; f < h.tns->num_filters; f++) put((uint64_t)(h.tns->rc_order[f] != 0), 1);
    put((uint64_t)(h.pitch_present != 0), 1);
    put((uint64_t)h.sns->ind_lf, 5);
    put((uint64_t)h.sns->ind_hf, 5);
    const bool submode_msb = (h.sns->shape_j >> 1) != 0;
    put((uint64_t)submode_msb, 1);
    put((uint64_t)(h.sns->gind >> LC3T_SNS_GAIN_LSB_BITS[h.sns->shape_j]), LC3T_SNS_GAIN_MSB_BITS[h.sns->shape_j]);
    put((uint64_t)(h.sns->ls_inda != 0), 1);
    if (!submode_msb) {
        put(h.sns->joint, 13);
        put(h.sns->joint >> 13, 12);
    } else {
        put(h.sns->joint, 12);
        put(h.sns->joint >> 12, 12);
    }
    if (h.pitch_present) {
        put((uint64_t)(h.ltpf_active != 0), 1);
        put((uint64_t)h.pitch_index, 9);
    }
    put((uint64_t)h.nf_factor, 3);
}

// BitstreamEncoding::encode :77-136 exactly as written (interleaved writes), one thread
__device__ __noinline__ void bitstream_encode_serial(const EncConfig& c, const SideHdr& h, const uint32_t* res_bits, int n_res,
                                                     const int16_t* xq, uint8_t* lsbs, uint8_t* out, int nbytes) {
    const QRes& q = *h.q;
    const TnsRes& tns = *h.tns;
    const int ne = c.ne, nbits = nbytes * 8;
    for (int i = 0; i < nbytes; i++) out[i] = 0;
    Writer w;
    w.buf = out;
    w.nbytes = nbytes;
    w.bp = 0;
    w.bp_side = nbytes - 1;
    w.mask_side = 1;
    auto put = [&](uint64_t v, int n) { w.uint_backward(v, n); };
    write_side_info(h, put);
    AcEnc st{0, 0x00ffffffu, -1, 0, 0};
    for (int f = 0; f < tns.num_filters; f++) {
        if (tns.rc_order[f] > 0) {
            ac_encode_serial(st, w, LC3T_AC_TNS_ORDER_CUMFREQ[tns.lpc_weighting][tns.rc_order[f] - 1],
                      LC3T_AC_TNS_ORDER_FREQ[tns.lpc_weighting][tns.rc_order[f] - 1]);
            for (int k = 0; k < tns.rc_order[f]; k++)
                ac_encode_serial(st, w, LC3T_AC_TNS_COEF_CUMFREQ[k][tns.rc_i[k + 8 * f]], LC3T_AC_TNS_COEF_FREQ[k][tns.rc_i[k + 8 * f]]);
        }
    }
    int nlsbs = 0;
    const int lsb_cap = 2 * ne;
    int cctx = 0;
    for (int k = 0; k < q.lastnz_trunc; k += 2) {
        int t = cctx + q.rate_flag + (k > ne / 2 ? 256 : 0);
        const int q0 = xq[k], q1 = xq[k + 1];
        uint32_t a = (uint32_t)(q0 < 0 ? -q0 : q0) & 0xffffu, a_lsb = a;
        uint32_t b = (uint32_t)(q1 < 0 ? -q1 : q1) & 0xffffu, b_lsb = b;
        int lev = 0;
        uint32_t lsb0 = 0, lsb1 = 0;
        while ((a > b ? a : b) >= 4) {
            const int pki = LC3T_AC_SPEC_LOOKUP[t + (lev < 3 ? lev : 3) * 1024];
            ac_encode_serial(st, w, LC3T_AC_SPEC_CUMFREQ[pki][16], LC3T_AC_SPEC_FREQ[pki][16]);
            if (q.lsb_mode && lev == 0) { lsb0 = a & 1; lsb1 = b & 1; }
            else { w.bool_backward((a & 1) == 1); w.bool_backward((b & 1) == 1); }
            a >>= 1;
            b >>= 1;
            lev++;
        }
        const int pki = LC3T_AC_SPEC_LOOKUP[t + (lev < 3 ? lev : 3) * 1024];
        const int sym = (int)(a + 4 * b);
        ac_encode_serial(st, w, LC3T_AC_SPEC_CUMFREQ[pki][sym], LC3T_AC_SPEC_FREQ[pki][sym]);
        if (q.lsb_mode && lev > 0) {
            a_lsb >>= 1;
            b_lsb >>= 1;
            if (nlsbs < lsb_cap) lsbs[nlsbs] = (uint8_t)lsb0;
            nlsbs++;
            if (a_lsb == 0 && q0 != 0) { if (nlsbs < lsb_cap) lsbs[nlsbs] = q0 > 0 ? 0 : 1; nlsbs++; }
            if (nlsbs < lsb_cap) lsbs[nlsbs] = (uint8_t)lsb1;
            nlsbs++;
            if (b_lsb == 0 && q1 != 0) { if (nlsbs < lsb_cap) lsbs[nlsbs] = q1 > 0 ? 0 : 1; nlsbs++; }
        }
        if (a_lsb > 0) w.bool_backward(q0 <= 0);
        if (b_lsb > 0) w.bool_backward(q1 <= 0);
        const int l = lev < 3 ? lev : 3;
        t = l <= 1 ? 1 + (int)(a + b) * (l + 1) : 12 + l;
        cctx = (cctx & 15) * 16 + t;
    }
    const int nbits_side = w.nbits_side_written(nbits);
    int nbits_ari = w.bp * 8;
    nbits_ari += 25 - (31 - __clz(st.range));
    nbits_ari += 8;                                   // QUIRK: `carry >= 0` is always true (:67)
    if (st.carry_count > 0) nbits_ari += st.carry_count * 8;
    int nres_enc = nbits - (nbits_side + nbits_ari);
    if (nres_enc < 0) nres_enc = 0;
    if (!q.lsb_mode) {
        for (int i = 0; i < n_res && i < nres_enc; i++) w.bool_backward((res_bits[i >> 5] >> (i & 31)) & 1u);
    } else {
        const int m = nres_enc < nlsbs ? nres_enc : nlsbs;
        for (int i = 0; i < m; i++) w.bool_backward(lsbs[i] == 1);
    }
    const int bits = ac_finish(st, w);
    if (st.carry_count > 0) {
        w.byte_forward((uint32_t)st.cache & 0xff);
        while (st.carry_count > 1) { w.byte_forward(0xff); st.carry_count -= 1; }
        w.uint_forward(0xffu >> (8 - bits), bits);
    } else {
        w.uint_forward((uint32_t)st.cache, bits);
    }
}

// forward byte sink of the fast path: every lane runs the same chain and stores the same byte (a lane-0-only store
// would split the warp and the rest of the symbol loop would issue twice)
struct FwdSink {
    uint8_t* buf;
    int nbytes, bp, lane;
    __device__ __forceinline__ void byte_forward(uint32_t v) {
        if (bp < nbytes) buf[bp] = (uint8_t)v;
        bp++;
    }
};

// append `n` bits (LSB first) to a little-endian bit array at position pos
__device__ __forceinline__ void bits_or(uint32_t* arr, int n_words, int pos, uint64_t val, int n) {
    if (n <= 0) return;
    const int w = pos >> 5, sh = pos & 31;
    const uint64_t v = (n < 64 ? (val & ((1ull << n) - 1ull)) : val) << sh;       // n <= 32 here
    if (w < n_words && (uint32_t)v != 0) atomicOr(&arr[w], (uint32_t)v);
    if (w + 1 < n_words && (uint32_t)(v >> 32) != 0) atomicOr(&arr[w + 1], (uint32_t)(v >> 32));
}

// Fast path of BitstreamEncoding::encode in three phases (enc_bitstream_kernel):
//   A  bs_prepare_w   one warp per frame: side information, symbol queue (TNS symbols first), side bits, deferred LSBs
//   B  ac_run_thread  one THREAD per frame: the range coder over the queue - a serial chain, so the frames of a CTA
//                     share one warp for it instead of each spending a whole warp's issue slots on it
//   C  bs_finish_w    one warp per frame: residual / LSB tail bits, collision test, merge of the two ends
struct AcJob {
    int nsym;          // queue length (TNS + spectral symbols); < 0: queue overflow, use the serial fallback
    int spos;          // side bits written so far (header + per-tuple bits)
    int nlsbs;         // deferred LSB entries (lsb_mode)
    int nbits_ari;     // out: bitstream_encoding.rs:63-73 forecast taken BEFORE ac_enc_finish
    int bp;            // out: forward bytes written, including ac_enc_finish
    int bits;          // out: valid bits of the final partial byte
    uint32_t last;     // out: value the final partial byte takes its top `bits` bits from
    int pad;
};

__device__ void bs_prepare_w(const EncConfig& c, const SideHdr& h, const int16_t* xq, uint32_t* side, int side_words,
                             uint32_t* tail, uint32_t* symq, int sym_cap, uint8_t* out, int out_words, AcJob* job, int lane) {
    const QRes& q = *h.q;
    const TnsRes& tns = *h.tns;
    const int ne = c.ne;
    WARP_STRIDE_R(i, side_words) side[i] = 0;
    WARP_STRIDE_R(i, out_words) ((uint32_t*)out)[i] = 0;
    if (q.lsb_mode) WARP_STRIDE_R(i, TAIL_WORDS) tail[i] = 0;
    __syncwarp();
    int spos = 0;
    {
        auto put = [&](uint64_t v, int n) {
            if (lane == 0) {
                const int w = spos >> 5, sh = spos & 31;
                const uint64_t vv = (v & ((1ull << n) - 1ull)) << sh;
                if (w < side_words) side[w] |= (uint32_t)vv;
                if (w + 1 < side_words) side[w + 1] |= (uint32_t)(vv >> 32);
            }
            spos += n;
        };
        write_side_info(h, put);
    }
    __syncwarp();
    // ---- per-tuple preparation: symbols -> queue, side bits and deferred LSBs -> bit arrays
    const uint32_t* xw = (const uint32_t*)xq;
    const int ntt = q.lastnz_trunc >> 1;
    const int CH = ntt > 0 ? (ntt + 31) >> 5 : 1;        // the tuples that exist, spread evenly over the lanes
    const int n0 = lane * CH;
    uint32_t cnt_a = 0, cnt_l = 0;                       // (symbols | side bits << 16), deferred LSB entries
    const int n1 = n0 + CH < ntt ? n0 + CH : ntt;
#pragma unroll 1
    for (int n = n0; n < n0 + CH; n++) if (n < n1) {
        const Tup t = tup_of(xw[n]);
        const bool defer = q.lsb_mode && t.L > 0;
        const uint32_t al = defer ? t.a0 >> 1 : t.a0, bl = defer ? t.b0 >> 1 : t.b0;
        const int sb = (defer ? 2 * (t.L - 1) : 2 * t.L) + (al > 0) + (bl > 0);
        cnt_a += (uint32_t)(t.L + 1) | ((uint32_t)sb << 16);
        if (defer) cnt_l += 2 + (al == 0 && t.q0 != 0) + (bl == 0 && t.q1 != 0);
    }
    const uint32_t inc_a = warp_incl_scan(cnt_a, lane), inc_l = warp_incl_scan(cnt_l, lane);
    const uint32_t tot_a = __shfl_sync(FULL, inc_a, 31);
    const int nlsbs = (int)__shfl_sync(FULL, inc_l, 31);
    int n_tns = 0;                                       // TNS symbols lead the queue (bitstream_encoding.rs:234-252)
    for (int f = 0; f < tns.num_filters; f++) if (tns.rc_order[f] > 0) n_tns += 1 + tns.rc_order[f];
    const int nsym = n_tns + (int)(tot_a & 0xffffu), nside_tup = (int)(tot_a >> 16);
    if (nsym > sym_cap) {
        if (lane == 0) job->nsym = -1;
        __syncwarp();
        return;
    }
    if (lane == 0) {
        int o = 0;
        for (int f = 0; f < tns.num_filters; f++) {
            if (tns.rc_order[f] > 0) {
                symq[o++] = (uint32_t)LC3T_AC_TNS_ORDER_CUMFREQ[tns.lpc_weighting][tns.rc_order[f] - 1] |
                            ((uint32_t)LC3T_AC_TNS_ORDER_FREQ[tns.lpc_weighting][tns.rc_order[f] - 1] << 16);
                for (int k = 0; k < tns.rc_order[f]; k++)
                    symq[o++] = (uint32_t)LC3T_AC_TNS_COEF_CUMFREQ[k][tns.rc_i[k + 8 * f]] | ((uint32_t)LC3T_AC_TNS_COEF_FREQ[k][tns.rc_i[k + 8 * f]] << 16);
            }
        }
    }
    {
        int so = n_tns + (int)((inc_a - cnt_a) & 0xffffu), bo = spos + (int)((inc_a - cnt_a) >> 16), lo = (int)(inc_l - cnt_l);
        int d2 = 0, d1 = 0;
        if (n0 >= 1 && n0 - 1 < ntt) d1 = tup_digit(tup_of(xw[n0 - 1]));
        if (n0 >= 2 && n0 - 2 < ntt) d2 = tup_digit(tup_of(xw[n0 - 2]));
#pragma unroll 1
        for (int n = n0; n < n0 + CH; n++) if (n < n1) {
            {
                const Tup t = tup_of(xw[n]);
                const int tc = d2 * 16 + d1 + q.rate_flag + (2 * n > ne / 2 ? 256 : 0);
                // escape levels (:262-283): one escape symbol per level from the model of min(lev, 3), and the level's
                // two magnitude bits (a, b interleaved) as side bits - except level 0 in lsb mode, whose bits are deferred
                const int L = t.L;
                const int pk0 = LC3T_AC_SPEC_LOOKUP[tc], pk1 = LC3T_AC_SPEC_LOOKUP[tc + 1024];
                const int pk2 = LC3T_AC_SPEC_LOOKUP[tc + 2048], pk3 = LC3T_AC_SPEC_LOOKUP[tc + 3072];
                auto esc = [&](int pk) { return (uint32_t)LC3T_AC_SPEC_CUMFREQ[pk][16] | ((uint32_t)LC3T_AC_SPEC_FREQ[pk][16] << 16); };
                if (L > 0) symq[so] = esc(pk0);
                if (L > 1) symq[so + 1] = esc(pk1);
                if (L > 2) symq[so + 2] = esc(pk2);
                if (L > 3) {
                    const uint32_t e3 = esc(pk3);
                    for (int lev = 3; lev < L; lev++) symq[so + lev] = e3;
                }
                so += L;
                const int skip = (q.lsb_mode && L > 0) ? 1 : 0;
                const uint32_t lsb0 = skip ? (t.a0 & 1u) : 0u, lsb1 = skip ? (t.b0 & 1u) : 0u;
                const uint32_t lm = (1u << (L - skip)) - 1u;                       // L - skip <= 14
                uint64_t sbits = (uint64_t)(spread_bits((t.a0 >> skip) & lm) | (spread_bits((t.b0 >> skip) & lm) << 1));
                int ns = 2 * (L - skip);
                const uint32_t a = t.a, b = t.b;
                const int pki = L == 0 ? pk0 : L == 1 ? pk1 : L == 2 ? pk2 : pk3;
                const int sym = (int)(a + 4 * b);
                symq[so++] = (uint32_t)LC3T_AC_SPEC_CUMFREQ[pki][sym] | ((uint32_t)LC3T_AC_SPEC_FREQ[pki][sym] << 16);
                uint32_t al = t.a0, bl = t.b0;
                if (q.lsb_mode && t.L > 0) {
                    al >>= 1;
                    bl >>= 1;
                    uint32_t lb = lsb0;
                    int nl = 1;
                    if (al == 0 && t.q0 != 0) { lb |= (uint32_t)(t.q0 > 0 ? 0 : 1) << nl; nl++; }
                    lb |= lsb1 << nl;
                    nl++;
                    if (bl == 0 && t.q1 != 0) { lb |= (uint32_t)(t.q1 > 0 ? 0 : 1) << nl; nl++; }
                    bits_or(tail, TAIL_WORDS, lo, lb, nl);
                    lo += nl;
                }
                if (al > 0) { sbits |= (uint64_t)(t.q0 <= 0) << ns; ns++; }
                if (bl > 0) { sbits |= (uint64_t)(t.q1 <= 0) << ns; ns++; }
                bits_or(side, side_words, bo, sbits, ns);
                bo += ns;
                d2 = d1;
                d1 = tup_digit(t);
            }
        }
    }
    spos += nside_tup;
    if (lane == 0) { job->nsym = nsym; job->spos = spos; job->nlsbs = nlsbs; }
    __syncwarp();
}

// Phase B: the range coder proper (bitstream_encoding.rs:234-352, 354-429), one thread per frame.
__device__ void ac_run_thread(const uint32_t* symq, uint8_t* out, int nbytes, AcJob* job) {
    const int nsym = job->nsym;
    if (nsym < 0) return;
    FwdSink w{out, nbytes, 0, 0};
    AcEnc st{0, 0x00ffffffu, -1, 0, 0};
    // Four symbols per round, the next four requested before the round starts: a frame's queue is this thread's own
    // stretch of global memory, so every load is a round trip of its own, and a one-symbol prefetch is consumed by the
    // register copy at the end of the very iteration that issued it (60 % of the kernel's stall samples sat there).
    // Reads run at most three entries past the queue's end, into the frame's forward-bytes area (values unused).
    uint32_t c0 = symq[0], c1 = symq[1], c2 = symq[2], c3 = symq[3];
    int i = 0;
#pragma unroll 1
    for (; i + 4 <= nsym; i += 4) {
        const uint32_t n0 = symq[i + 4], n1 = symq[i + 5], n2 = symq[i + 6], n3 = symq[i + 7];
        ac_encode(st, w, (int)(c0 & 0xffffu), (int)(c0 >> 16));
        ac_encode(st, w, (int)(c1 & 0xffffu), (int)(c1 >> 16));
        ac_encode(st, w, (int)(c2 & 0xffffu), (int)(c2 >> 16));
        ac_encode(st, w, (int)(c3 & 0xffffu), (int)(c3 >> 16));
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    }
    if (i < nsym) ac_encode(st, w, (int)(c0 & 0xffffu), (int)(c0 >> 16));
    if (i + 1 < nsym) ac_encode(st, w, (int)(c1 & 0xffffu), (int)(c1 >> 16));
    if (i + 2 < nsym) ac_encode(st, w, (int)(c2 & 0xffffu), (int)(c2 >> 16));
    int nbits_ari = w.bp * 8;
    nbits_ari += 25 - (31 - __clz(st.range));
    nbits_ari += 8;                                   // QUIRK: `carry >= 0` is always true (:67)
    if (st.carry_count > 0) nbits_ari += st.carry_count * 8;
    job->nbits_ari = nbits_ari;
    const int bits = ac_finish(st, w);                // the tail bits written in between never touch the coder's state
    uint32_t last;
    if (st.carry_count > 0) {
        w.byte_forward((uint32_t)st.cache & 0xff);
        while (st.carry_count > 1) { w.byte_forward(0xff); st.carry_count -= 1; }
        last = 0xffu >> (8 - bits);
    } else {
        last = (uint32_t)st.cache;
    }
    job->bp = w.bp;
    job->bits = bits;
    job->last = last;
}

// Phase C: residual / LSB bits behind the side stream, collision test, final partial byte.  Returns false when the two
// ends of the frame meet or the queue overflowed (caller falls back to the reference-order writer).
__device__ bool bs_finish_w(const QRes& q, int n_res, uint32_t* side, int side_words, const uint32_t* tail, uint8_t* out,
                            int nbytes, const AcJob* job, int lane) {
    if (job->nsym < 0) return false;
    const int nbits = nbytes * 8;
    int spos = job->spos;
    int nres_enc = nbits - (spos + job->nbits_ari);
    if (nres_enc < 0) nres_enc = 0;
    const int nlsbs = job->nlsbs;
    const int m = q.lsb_mode ? (nres_enc < nlsbs ? nres_enc : nlsbs) : (n_res < nres_enc ? n_res : nres_enc);
    if (lane < TAIL_WORDS) {                          // tail bits [0, m) -> side stream at spos
        const int lo = lane * 32;
        if (lo < m) {
            const int n = m - lo < 32 ? m - lo : 32;
            bits_or(side, side_words, spos + lo, tail[lane], n);
        }
    }
    spos += m;
    const int bp = job->bp, bits = job->bits;
    if (bp >= nbytes || 8 * bp + bits + spos > nbits) return false;
    __syncwarp();
    if (lane == 0) out[bp] |= (uint8_t)(job->last & (0xff00u >> bits) & 0xffu);
    __syncwarp();
    return true;
}

// hand-off record between the three kernels of this file (int32 words per stream)
enum {
    QH_BW = 0, QH_NBITS_BW, QH_IND_LF, QH_IND_HF, QH_SHAPE_J, QH_GIND, QH_LS_INDA, QH_LS_INDB, QH_JOINT_LO, QH_JOINT_HI,
    QH_NBITS_TNS, QH_LPC_WEIGHTING, QH_NUM_FILTERS, QH_ORDER0, QH_ORDER1, QH_PAD0,
    QH_RC_I = 16,
    QH_GG_IND = 32, QH_NBITS_SPEC, QH_NBITS_LSB, QH_NBITS_TRUNC, QH_LSB_MODE, QH_RATE_FLAG, QH_LASTNZ_TRUNC, QH_GG,
};
static_assert(QH_GG < QH_WORDS, "hand-off record too small");

// Kernel A1: bandwidth detector and SNS.  Spectrum in place in global memory, decisions into the hand-off record.
// Four frames per CTA here: the warps of a CTA wait at the pulse-search barriers, and with eight of them the wait showed.
constexpr int SNS_WARPS = 4;
__global__ void __launch_bounds__(SNS_WARPS * 32) enc_sns_kernel(QuantParams p) {
    extern __shared__ __align__(16) uint8_t smem[];
    const EncConfig& c = *p.cfg;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int stream = blockIdx.x * SNS_WARPS + wib;
    if (stream >= p.n_streams) return;                            // the warps that stay meet at named barriers sized for them
    const int ne = c.ne;
    float* xf = (float*)(smem + (size_t)wib * (sizeof(float) * (NE_MAX + S_FLOATS)));   // [NE_MAX]
    float* S = xf + NE_MAX;                                                             // [S_FLOATS]
    float4* gx = (float4*)(p.xf + (size_t)stream * ne);
    WARP_STRIDE_R(i, ne / 4) ((float4*)xf)[i] = gx[i];
    const float* eb = p.e_b + (size_t)stream * 64;
    S[lane] = eb[lane];
    S[lane + 32] = eb[lane + 32];
    __syncwarp();
    const int32_t* eh = p.ehand + (size_t)stream * EH_WORDS;
    const BwRes bw = bandwidth_detect(c, S);
    const SnsRes sns = sns_encode_w(c, xf, S, eh[EH_ATTACK] != 0, lane, wib, min(SNS_WARPS, p.n_streams - blockIdx.x * SNS_WARPS));
    WARP_STRIDE_R(i, ne / 4) gx[i] = ((const float4*)xf)[i];
    int32_t* qh = p.qhand + (size_t)stream * QH_WORDS;
    if (lane == 0) {
        qh[QH_BW] = bw.bw; qh[QH_NBITS_BW] = bw.nbits;
        qh[QH_IND_LF] = sns.ind_lf; qh[QH_IND_HF] = sns.ind_hf; qh[QH_SHAPE_J] = sns.shape_j; qh[QH_GIND] = sns.gind;
        qh[QH_LS_INDA] = sns.ls_inda; qh[QH_LS_INDB] = sns.ls_indb;
        qh[QH_JOINT_LO] = (int32_t)(uint32_t)sns.joint; qh[QH_JOINT_HI] = (int32_t)(uint32_t)(sns.joint >> 32);
    }
}

// Kernel A2: TNS analysis and filtering.
__global__ void __launch_bounds__(QNT_THREADS, 4) enc_tns_kernel(QuantParams p) {
    extern __shared__ __align__(16) uint8_t smem[];
    const EncConfig& c = *p.cfg;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int stream = blockIdx.x * QW + wib;
    if (stream >= p.n_streams) return;
    const int ne = c.ne;
    float* xf = (float*)(smem + (size_t)wib * (sizeof(float) * (NE_MAX + S_FLOATS)));   // [NE_MAX]
    float* S = xf + NE_MAX;                                                             // [S_FLOATS]
    float4* gx = (float4*)(p.xf + (size_t)stream * ne);
    WARP_STRIDE(i, ne / 4) ((float4*)xf)[i] = gx[i];
    __syncwarp();
    const int32_t* eh = p.ehand + (size_t)stream * EH_WORDS;
    int32_t* qh = p.qhand + (size_t)stream * QH_WORDS;
    TnsRes tns;
    tns_encode_w(c, xf, S, qh[QH_BW], p.nbytes * 8, eh[EH_NEAR_NYQUIST] != 0, tns, lane);
    if (tns.rc_order[0] != 0 || tns.rc_order[1] != 0) {           // the spectrum only changes when a filter is active
        WARP_STRIDE(i, ne / 4) gx[i] = ((const float4*)xf)[i];
    }
    if (lane == 0) {
        qh[QH_NBITS_TNS] = tns.nbits_tns; qh[QH_LPC_WEIGHTING] = tns.lpc_weighting; qh[QH_NUM_FILTERS] = tns.num_filters;
        qh[QH_ORDER0] = tns.rc_order[0]; qh[QH_ORDER1] = tns.rc_order[1];
    }
    if (lane < 16) qh[QH_RC_I + lane] = tns.rc_i[lane];
}

// Kernel B: SpectralQuantization::run.  Shaped spectrum -> quantised spectrum + gain decisions.  One frame per warp
// (lc3b_encode_frames; IDS: lc3b_encode_frames_subset), or, WALK (always with IDS: a row's state row comes from the row
// table), a warp per row of a time-parallel call's row table walking the row's frames in order, the rate loop's offsets
// (ES_Q_*) carrying from one frame to the next.  The walk is a separate instantiation, so the frame-by-frame path keeps
// its registers.  As in enc_ltpf_kernel the table is sorted by count, descending: the warps that still have frame f are
// warps 0 .. n_live - 1 (n_live = the CTA's rows with count > f, recounted every frame), the barriers count exactly them
// and warp 0 does the ordered sums of lanes < n_live.
template <bool WALK, bool IDS>
__global__ void __launch_bounds__(QNT_THREADS) enc_quantize_kernel(QuantParams p) {
    extern __shared__ __align__(16) uint8_t smem[];
    const EncConfig& c = *p.cfg;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int stream = blockIdx.x * QW + wib;
    if (stream >= p.n_streams) return;
    const int ne = c.ne;
    uint8_t* wb = smem + (size_t)wib * QUANTIZE_WARP_BYTES;
    float* xf = (float*)wb;                                       // [NE_MAX]
    float* e4 = xf + NE_MAX;                                      // [100]
    float* T = e4 + 100;                                          // [224]
    int16_t* xq = (int16_t*)(T + 224);                            // [NE_MAX]
    static_assert(!WALK || IDS, "the row walk addresses state through the row table");
    const RowSpan rs = WALK ? row_span(p.rows, stream) : RowSpan{state_row<IDS>(p.ids, stream), stream, 1};
    int32_t* es = p.estate + (size_t)rs.row * ES_WORDS;
    const int n_cta = min(QW, p.n_streams - blockIdx.x * QW);     // warps of this CTA that have a frame
    const int cnt = WALK && lane < n_cta ? row_span(p.rows, blockIdx.x * QW + lane).count : 0;   // lane j: warp j's
    const int F = WALK ? __reduce_max_sync(0xffffffffu, rs.count) : 1;   // uniform registers, see enc_ltpf_kernel
    for (int f = 0; f < F; f++) {
        const int n_live = WALK ? (int)__reduce_add_sync(0xffffffffu, cnt > f ? 1u : 0u) : n_cta;
        const size_t unit = (size_t)rs.off + f;
        const float4* gx = (const float4*)(p.xf + unit * ne);
        WARP_STRIDE(i, ne / 4) ((float4*)xf)[i] = gx[i];
        __syncwarp();
        const int32_t* eh = p.ehand + unit * EH_WORDS;
        int32_t* qh = p.qhand + unit * QH_WORDS;
        const QRes q = spectral_quantization_w(c, es, xf, xq, e4, T, p.nbytes * 8, qh[QH_NBITS_BW], qh[QH_NBITS_TNS], eh[EH_NBITS_LTPF],
                                               lane, wib, n_live, smem);
        uint32_t* gq = (uint32_t*)(p.xq + unit * ne);
        WARP_STRIDE(i, ne / 2) gq[i] = ((const uint32_t*)xq)[i];
        if (lane == 0) {
            qh[QH_GG_IND] = q.gg_ind; qh[QH_NBITS_SPEC] = q.nbits_spec; qh[QH_NBITS_LSB] = q.nbits_lsb; qh[QH_NBITS_TRUNC] = q.nbits_trunc;
            qh[QH_LSB_MODE] = q.lsb_mode; qh[QH_RATE_FLAG] = q.rate_flag; qh[QH_LASTNZ_TRUNC] = q.lastnz_trunc;
            qh[QH_GG] = (int32_t)__float_as_uint(q.gg);
        }
        if (WALK) __syncwarp();                                   // lane 0's state update before the next frame reads it
    }
}

// Bitstream stage = three kernels.  The per-stream hand-off lives in EncoderState::bs_scratch:
//   [ job (8 words) | tail bits (TAIL_WORDS) | side bits (side_words) | symbol queue (sym_cap + 1) | forward bytes (out_words) ]
// C1 enc_bs_prepare_kernel   warp per frame: residual bits, noise factor, side information, symbol queue, side bits
// C2 enc_range_coder_kernel  THREAD per frame: the range coder is one serial chain per frame, so frames are the only
//                            parallel axis; a warp per frame spent 6 k of its 12.8 k issue slots repeating it in 32 lanes
// C3 enc_bs_finish_kernel    warp per frame: tail bits, collision test, merge of the two ends, coalesced output
struct BsLayout { int job, tail, side, symq, fwd, words; };
__host__ __device__ inline BsLayout bs_layout(int side_words, int sym_cap, int out_words) {
    BsLayout L;
    L.job = 0;
    L.tail = 8;
    L.side = L.tail + TAIL_WORDS;
    L.symq = L.side + side_words;
    L.fwd = L.symq + sym_cap + 1;
    L.words = L.fwd + out_words;
    return L;
}
static_assert(sizeof(AcJob) == 32, "AcJob is 8 words");

__device__ __forceinline__ void load_results(const QuantParams& p, int stream, BwRes& bw, SnsRes& sns, TnsRes& tns, QRes& q,
                                             SideHdr& h, int* rc_i, int lane) {
    const int32_t* qh = p.qhand + (size_t)stream * QH_WORDS;
    const int32_t* eh = p.ehand + (size_t)stream * EH_WORDS;
    if (lane < 16) rc_i[lane] = qh[QH_RC_I + lane];
    bw = BwRes{qh[QH_BW], qh[QH_NBITS_BW]};
    sns.ind_lf = qh[QH_IND_LF]; sns.ind_hf = qh[QH_IND_HF]; sns.shape_j = qh[QH_SHAPE_J]; sns.gind = qh[QH_GIND];
    sns.ls_inda = qh[QH_LS_INDA]; sns.ls_indb = qh[QH_LS_INDB];
    sns.joint = (uint64_t)(uint32_t)qh[QH_JOINT_LO] | ((uint64_t)(uint32_t)qh[QH_JOINT_HI] << 32);
    tns.nbits_tns = qh[QH_NBITS_TNS]; tns.lpc_weighting = qh[QH_LPC_WEIGHTING]; tns.num_filters = qh[QH_NUM_FILTERS];
    tns.rc_order[0] = qh[QH_ORDER0]; tns.rc_order[1] = qh[QH_ORDER1];
    tns.rc_i = rc_i;
    q.gg_ind = qh[QH_GG_IND]; q.nbits_spec = qh[QH_NBITS_SPEC]; q.nbits_lsb = qh[QH_NBITS_LSB]; q.nbits_trunc = qh[QH_NBITS_TRUNC];
    q.lsb_mode = qh[QH_LSB_MODE]; q.rate_flag = qh[QH_RATE_FLAG]; q.lastnz_trunc = qh[QH_LASTNZ_TRUNC];
    q.gg = __uint_as_float((uint32_t)qh[QH_GG]);
    h.bw = &bw; h.sns = &sns; h.tns = &tns; h.q = &q;
    h.pitch_present = eh[EH_PITCH_PRESENT]; h.ltpf_active = eh[EH_LTPF_ACTIVE]; h.pitch_index = eh[EH_PITCH_INDEX];
    h.lg = 0;
    while ((1 << h.lg) < p.cfg->ne / 2) h.lg++;
}

__global__ void __launch_bounds__(QNT_THREADS) enc_bs_prepare_kernel(QuantParams p) {
    extern __shared__ __align__(16) uint8_t smem[];
    const EncConfig& c = *p.cfg;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int stream = blockIdx.x * QW + wib;
    if (stream >= p.n_streams) return;                            // warps are independent: no CTA-wide barrier below
    const int ne = c.ne;
    uint8_t* wb = smem + (size_t)wib * p.w_bytes;
    float* xf = (float*)wb;                                       // [NE_MAX]
    int16_t* xq = (int16_t*)(xf + NE_MAX);                        // [NE_MAX]
    int* rc_i = (int*)(xq + NE_MAX);                              // [16]
    AcJob* job = (AcJob*)(rc_i + 16);                             // 8 words
    uint32_t* tail = (uint32_t*)(job + 1);                        // [TAIL_WORDS]
    uint32_t* side = tail + TAIL_WORDS;                           // [side_words]
    uint32_t* symq = side + p.side_words;                         // [sym_cap + 1]
    uint8_t* out = (uint8_t*)(symq + p.sym_cap + 1);              // [out_words * 4] (zeroed here, filled by the range coder kernel)
    {
        const float4* gx = (const float4*)(p.xf + (size_t)stream * ne);
        // (the kernel's first loads stay unrolled: all of them in flight at once)
        WARP_STRIDE(i, ne / 4) ((float4*)xf)[i] = gx[i];
        const uint32_t* gq = (const uint32_t*)(p.xq + (size_t)stream * ne);
        WARP_STRIDE(i, ne / 2) ((uint32_t*)xq)[i] = gq[i];
        if (lane < TAIL_WORDS) tail[lane] = 0;
    }
    BwRes bw;
    SnsRes sns;
    TnsRes tns;
    QRes q;
    SideHdr h;
    load_results(p, stream, bw, sns, tns, q, h, rc_i, lane);
    __syncwarp();
    int n_res = 0;
    if (!q.lsb_mode) n_res = residual_bits_w(ne, xf, xq, q.gg, q.nbits_spec - q.nbits_trunc + 4, tail, lane);
    __syncwarp();
    h.nf_factor = noise_factor_w(c, xf, xq, bw.bw, q.gg, lane, wib, min(QW, p.n_streams - blockIdx.x * QW), (size_t)p.w_bytes);
    bs_prepare_w(c, h, xq, side, p.side_words, tail, symq, p.sym_cap, out, p.out_words, job, lane);
    if (lane == 0) { job->pad = n_res | (h.nf_factor << 16); }
    __syncwarp();
    // hand-off: job | tail | side | queue (only the used part) are contiguous in the warp's slice
    const BsLayout L = bs_layout(p.side_words, p.sym_cap, p.out_words);
    uint32_t* g = p.bs_scratch + (size_t)stream * p.bs_words;
    const int nq = job->nsym < 0 ? 0 : job->nsym + 1;
    const uint32_t* src = (const uint32_t*)job;
    WARP_STRIDE_R(i, L.symq + nq) g[i] = src[i];
    WARP_STRIDE_R(i, p.out_words) g[L.fwd + i] = 0;
}

__global__ void __launch_bounds__(128) enc_range_coder_kernel(QuantParams p) {
    const int stream = blockIdx.x * 128 + threadIdx.x;
    if (stream >= p.n_streams) return;
    const BsLayout L = bs_layout(p.side_words, p.sym_cap, p.out_words);
    uint32_t* g = p.bs_scratch + (size_t)stream * p.bs_words;
    ac_run_thread(g + L.symq, (uint8_t*)(g + L.fwd), p.nbytes, (AcJob*)g);
}

__global__ void __launch_bounds__(QNT_THREADS) enc_bs_finish_kernel(QuantParams p) {
    extern __shared__ __align__(16) uint8_t smem[];
    const EncConfig& c = *p.cfg;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int stream = blockIdx.x * QW + wib;
    if (stream >= p.n_streams) return;
    const int ne = c.ne, nbytes = p.nbytes;
    const BsLayout L = bs_layout(p.side_words, p.sym_cap, p.out_words);
    // warp slice: job | tail | side | forward bytes | rc_i | xq (fallback only)
    uint32_t* wbase = (uint32_t*)(smem + (size_t)wib * p.w_bytes_fin);
    AcJob* job = (AcJob*)wbase;
    uint32_t* tail = wbase + L.tail;
    uint32_t* side = wbase + L.side;
    uint8_t* out = (uint8_t*)(wbase + L.symq);
    int* rc_i = (int*)(wbase + L.symq + p.out_words);
    int16_t* xq = (int16_t*)(rc_i + 16);
    const uint32_t* g = p.bs_scratch + (size_t)stream * p.bs_words;
    WARP_STRIDE(i, L.symq) wbase[i] = g[i];                          // unrolled: the loads of a slice go out together
    WARP_STRIDE(i, p.out_words) ((uint32_t*)out)[i] = g[L.fwd + i];
    BwRes bw;
    SnsRes sns;
    TnsRes tns;
    QRes q;
    SideHdr h;
    load_results(p, stream, bw, sns, tns, q, h, rc_i, lane);
    __syncwarp();
    const int n_res = job->pad & 0xffff;
    h.nf_factor = job->pad >> 16;
    if (p.inline_ac) {                                             // every lane runs the same chain and stores the same bytes
        ac_run_thread(g + L.symq, out, nbytes, job);
        __syncwarp();
    }
    const bool ok = bs_finish_w(q, n_res, side, p.side_words, tail, out, nbytes, job, lane);
    uint8_t* dst = p.frames_out + (size_t)stream * p.frame_stride;
    if (ok) {
        WARP_STRIDE_R(b, nbytes) {
            const int i = nbytes - 1 - b;
            dst[b] = out[b] | (uint8_t)(side[i >> 2] >> (8 * (i & 3)));
        }
    } else {                                                       // reference-order rewrite of the whole frame by one lane
        const uint32_t* gq = (const uint32_t*)(p.xq + (size_t)stream * ne);
        WARP_STRIDE_R(i, ne / 2) ((uint32_t*)xq)[i] = gq[i];
        __syncwarp();
        if (lane == 0) bitstream_encode_serial(c, h, tail, n_res, xq, p.lsbs + (size_t)stream * 2 * ne, out, nbytes);
        __syncwarp();
        WARP_STRIDE_R(b, nbytes) dst[b] = out[b];
    }
}

static void bitstream_sizes(int ne, int nbytes, int* side_words, int* sym_cap, int* out_words) {
    const int nbits = nbytes * 8;
    *side_words = (nbits + 31) / 32 + 2;
    *sym_cap = ne / 2 + nbits / 2 + 32 + 18;   // tuples + escapes the truncation rule can admit (2 bits each at least) + TNS
    *out_words = (nbytes + 3) / 4 + 1;
}
int enc_bitstream_scratch_words(int ne, int max_nbytes) {
    int sw, sc, ow;
    bitstream_sizes(ne, max_nbytes, &sw, &sc, &ow);
    return bs_layout(sw, sc, ow).words;
}
// shared-memory slice of one warp in the prepare kernel / the finish kernel
static size_t bitstream_warp_bytes(int ne, int nbytes, QuantParams* p) {
    int side_words, sym_cap, out_words;
    bitstream_sizes(ne, nbytes, &side_words, &sym_cap, &out_words);
    size_t wbytes = sizeof(float) * NE_MAX + sizeof(int16_t) * NE_MAX + sizeof(int) * 16 + sizeof(AcJob) +
                    sizeof(uint32_t) * (size_t)(TAIL_WORDS + side_words + sym_cap + 1 + out_words);
    wbytes = (wbytes + 15) & ~(size_t)15;
    size_t fbytes = sizeof(uint32_t) * (size_t)(8 + TAIL_WORDS + side_words + out_words + 16) + sizeof(int16_t) * NE_MAX;
    fbytes = (fbytes + 15) & ~(size_t)15;
    if (p) {
        p->side_words = side_words; p->sym_cap = sym_cap; p->out_words = out_words;
        p->w_bytes = (int)wbytes; p->w_bytes_fin = (int)fbytes;
    }
    return wbytes;
}
constexpr size_t SHAPE_SMEM = QW * sizeof(float) * (NE_MAX + S_FLOATS);
constexpr size_t QUANTIZE_SMEM = QW * QUANTIZE_WARP_BYTES;

// dynamic shared memory limits, once per handle (lc3b_encoder_init) for the largest frame the handle accepts
cudaError_t prepare_enc_quant(const EncoderState& st) {
    cudaError_t e = cudaFuncSetAttribute(enc_sns_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(SHAPE_SMEM / QW * SNS_WARPS));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(enc_tns_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SHAPE_SMEM);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(enc_quantize_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)QUANTIZE_SMEM);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(enc_quantize_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)QUANTIZE_SMEM);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(enc_quantize_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)QUANTIZE_SMEM);
    if (e == cudaSuccess)
        e = cudaFuncSetAttribute(enc_bs_prepare_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)(QW * bitstream_warp_bytes(st.cfg.ne, st.max_nbytes, nullptr)));
    return e;
}

void plan_enc_quant(LaunchPlan& plan, const EncoderState& st, uint8_t* frames_out, int nbytes, size_t frame_stride, int stages,
                    const int32_t* ids, const int32_t* rows, int n_rows) {
    QuantParams p;
    memset(&p, 0, sizeof(p));
    p.cfg = st.ecfg;
    p.n_streams = st.n_streams;
    p.nbytes = nbytes;
    p.frame_stride = frame_stride;
    p.xf = st.xf;
    p.e_b = st.e_b;
    p.ehand = st.ehand;
    p.estate = st.estate;
    p.xq = st.xq;
    p.qhand = st.qhand;
    p.lsbs = st.lsbs;
    p.bs_scratch = st.bs_scratch;
    p.bs_words = st.bs_words;
    p.inline_ac = 0;
    p.frames_out = frames_out;
    p.ids = ids;
    p.rows = rows;
    const size_t wbytes = bitstream_warp_bytes(st.cfg.ne, nbytes, &p);
    const int grid = (p.n_streams + QW - 1) / QW;
    if (stages & 1) plan.add(enc_sns_kernel, (unsigned)((p.n_streams + SNS_WARPS - 1) / SNS_WARPS), SNS_WARPS * 32, SHAPE_SMEM / QW * SNS_WARPS, p);
    if (stages & 2) plan.add(enc_tns_kernel, (unsigned)grid, QNT_THREADS, SHAPE_SMEM, p);
    if (stages & 4) {                                              // one warp per frame, or per row walking its frames
        QuantParams pw = p;
        if (rows) pw.n_streams = n_rows;
        plan.add(rows ? enc_quantize_kernel<true, true> : ids ? enc_quantize_kernel<false, true> : enc_quantize_kernel<false, false>,
                 (unsigned)((pw.n_streams + QW - 1) / QW), QNT_THREADS, QUANTIZE_SMEM, pw);
    }
    if (stages & 8) {
        plan.add(enc_bs_prepare_kernel, (unsigned)grid, QNT_THREADS, QW * wbytes, p);
        // a thread-per-frame kernel needs ~12 k frames before its serial latency (~80 us) is amortised
        p.inline_ac = p.n_streams < 12288 ? 1 : 0;
        if (!p.inline_ac) plan.add(enc_range_coder_kernel, (unsigned)((p.n_streams + 127) / 128), 128, 0, p);
        plan.add(enc_bs_finish_kernel, (unsigned)grid, QNT_THREADS, QW * (size_t)p.w_bytes_fin, p);
    }
}

}  // namespace lc3b
