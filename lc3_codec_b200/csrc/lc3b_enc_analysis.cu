// lc3b engine, encoder kernels 1-2 of 6: PCM -> MDCT spectrum + band energies (enc_mdct_kernel), attack flag + LTPF
// parameters (enc_ltpf_kernel).  One WARP per frame.  Two kernels so each one's code stays near the SM's instruction cache.  Compiled with -fmad=false: every expression below rounds exactly like the reference's f32 code.
//
// Replaces, per stream, the first half of EncoderChannel::encode (src/encoder/lc3_encoder.rs:63-90):
//   ModDiscreteCosTrans::run     src/encoder/modified_dct.rs:108 (time buffer :126, window+fold :73, DCT-IV
//                                src/common/dct_iv.rs:49 over src/common/kissfft.rs:78, energies :140, near-Nyquist :154)
//   AttackDetector::run          src/encoder/attack_detector.rs:45
//   LongTermPostFilter::run      src/encoder/long_term_post_filter.rs:139 (resampler, 50 Hz high-pass, pitch detection,
//                                pitch-lag parameter, activation bit)
// Parallelisation never reassociates a sum: each lane owns whole outputs (one band energy, one resampled sample, one
// correlation lag, one butterfly) and accumulates them in the reference's order; only truly serial recurrences (the
// biquad, the block-energy envelope, the decision logic) run on lane 0.  The FFT is kissfft's own decimation-in-time
// schedule (same factor order 4,4,..,2,3,5, same butterflies, same twiddle products) executed level by level with
// the butterflies of a level spread over the lanes, so the spectrum is bit-identical to the reference's.
#include <string.h>

#include "lc3b_enc_common.cuh"
#include "lc3b_plan.cuh"
#include "lc3b_math.cuh"
#include "lc3_tables.h"

namespace lc3b {

struct AnalysisParams {
    const EncConfig* cfg;
    const float* win;
    const float2* dtw;
    const float2* ftw;
    const int32_t* perm;
    const int16_t* pcm;
    size_t pcm_stride;
    int nbytes;
    int n_streams;
    int16_t* thist;
    int16_t* xs_hist;
    float* x12;
    float* x6;
    int32_t* estate;
    float* xf;
    float* e_b;
    int32_t* ehand;
    int smem_per_warp;
    const int32_t* ids;   // subset call: row u is handle stream ids[u] (the one-frame IDS instantiations only)
    const int32_t* rows;  // time-parallel call: the row table (lc3b_common.cuh), n_streams its rows (enc_ltpf_kernel<true, true>)
};

constexpr int ANA_WARPS = 4;

struct C2 { float r, i; };
__device__ __forceinline__ C2 cmul(C2 a, C2 b) { return {a.r * b.r - a.i * b.i, a.r * b.i + a.i * b.r}; }   // complex.rs:16-24
__device__ __forceinline__ C2 cadd(C2 a, C2 b) { return {a.r + b.r, a.i + b.i}; }
__device__ __forceinline__ C2 csub(C2 a, C2 b) { return {a.r - b.r, a.i - b.i}; }
__device__ __forceinline__ C2 ld(const float2* p, int i) { float2 v = p[i]; return {v.x, v.y}; }
__device__ __forceinline__ C2 lds(const C2* p, int i) { return p[i]; }

// kissfft.rs:133-256, one butterfly (index u of a block `f` with sub-length m) per call
__device__ __forceinline__ void bfly2(C2* f, const float2* tw, int fs, int m, int u) {
    C2 t = cmul(f[m + u], ld(tw, u * fs));
    f[m + u] = csub(f[u], t);
    f[u] = cadd(f[u], t);
}
__device__ __forceinline__ void bfly4(C2* f, const float2* tw, int fs, int m, int u) {
    const int m2 = 2 * m, m3 = 3 * m;
    C2 s0 = cmul(f[u + m], ld(tw, u * fs));
    C2 s1 = cmul(f[u + m2], ld(tw, u * fs * 2));
    C2 s2 = cmul(f[u + m3], ld(tw, u * fs * 3));
    C2 s5 = csub(f[u], s1);
    C2 f0 = cadd(f[u], s1);
    C2 s3 = cadd(s0, s2);
    C2 s4 = csub(s0, s2);
    f[u + m2] = csub(f0, s3);
    f[u] = cadd(f0, s3);
    f[u + m] = {s5.r + s4.i, s5.i - s4.r};             // forward transform (inverse == false)
    f[u + m3] = {s5.r - s4.i, s5.i + s4.r};
}
__device__ __forceinline__ void bfly3(C2* f, const float2* tw, int fs, int m, int u) {
    const int m2 = 2 * m;
    const C2 epi3 = ld(tw, fs * m);
    C2 s1 = cmul(f[u + m], ld(tw, u * fs));
    C2 s2 = cmul(f[u + m2], ld(tw, u * fs * 2));
    C2 s3 = cadd(s1, s2);
    C2 s0 = csub(s1, s2);
    C2 fi = f[u];
    C2 fm = {fi.r - (s3.r * 0.5f), fi.i - (s3.i * 0.5f)};
    s0.r *= epi3.i;
    s0.i *= epi3.i;
    f[u] = cadd(fi, s3);
    f[u + m2] = {fm.r + s0.i, fm.i - s0.r};
    f[u + m] = {fm.r - s0.i, fm.i + s0.r};
}
__device__ __forceinline__ void bfly5(C2* f, const float2* tw, int fs, int m, int u) {
    const C2 ya = ld(tw, fs * m), yb = ld(tw, fs * 2 * m);
    const int m1 = m, m2 = 2 * m, m3 = 3 * m, m4 = 4 * m;
    C2 s0 = f[u];
    C2 s1 = cmul(f[u + m1], ld(tw, u * fs));
    C2 s2 = cmul(f[u + m2], ld(tw, u * 2 * fs));
    C2 s3 = cmul(f[u + m3], ld(tw, u * 3 * fs));
    C2 s4 = cmul(f[u + m4], ld(tw, u * 4 * fs));
    C2 s7 = cadd(s1, s4), s10 = csub(s1, s4), s8 = cadd(s2, s3), s9 = csub(s2, s3);
    C2 f0;
    f0.r = s0.r + (s7.r + s8.r);
    f0.i = s0.i + (s7.i + s8.i);
    f[u] = f0;
    C2 s5 = {s0.r + (s7.r * ya.r) + (s8.r * yb.r), s0.i + (s7.i * ya.r) + (s8.i * yb.r)};
    C2 s6 = {(s10.i * ya.i) + (s9.i * yb.i), -(s10.r * ya.i) - (s9.r * yb.i)};
    f[u + m1] = csub(s5, s6);
    f[u + m4] = cadd(s5, s6);
    C2 s11 = {s0.r + (s7.r * yb.r) + (s8.r * ya.r), s0.i + (s7.i * yb.r) + (s8.i * ya.r)};
    C2 s12 = {-(s10.i * yb.i) + (s9.i * ya.i), (s10.r * yb.i) - (s9.r * ya.i)};
    f[u + m2] = cadd(s11, s12);
    f[u + m3] = csub(s11, s12);
}

template <bool IDS>
__global__ void __launch_bounds__(ANA_WARPS * 32) enc_mdct_kernel(AnalysisParams p) {
    extern __shared__ __align__(16) uint8_t smem[];
    const EncConfig& c = *p.cfg;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int stream = blockIdx.x * ANA_WARPS + wid;             // the call's row; only the time history is per stream
    if (stream >= p.n_streams) return;
    const int nf = c.nf, ne = c.ne, z = c.z, N = c.n_fft, half = nf / 2;

    uint8_t* base = smem + (size_t)wid * p.smem_per_warp;
    float* wk = (float*)base;                       // nf floats
    C2* cx = (C2*)(wk + nf);                        // N complex
    int16_t* tb = (int16_t*)(cx + N);               // 2*nf

    const int16_t* in = p.pcm + (size_t)stream * p.pcm_stride;
    int16_t* thist = p.thist + (size_t)state_row<IDS>(p.ids, stream) * (nf - z);

    // ---- update_time_buffer (modified_dct.rs:126-138)
    // samples move two at a time: nf, z and nf - z are even, the history rows are 4-byte aligned, the input row usually is
    WARP_STRIDE(n, (nf - z) / 2) ((uint32_t*)tb)[n] = ((const uint32_t*)thist)[n];
    if (((uintptr_t)in & 3) == 0) { WARP_STRIDE(n, nf / 2) ((uint32_t*)(tb + nf - z))[n] = ((const uint32_t*)in)[n]; }
    else { WARP_STRIDE(n, nf) tb[nf - z + n] = in[n]; }
    WARP_STRIDE(n, z / 2) ((uint32_t*)(tb + 2 * nf - z))[n] = 0u;
    __syncwarp();
    WARP_STRIDE(n, (nf - z) / 2) ((uint32_t*)thist)[n] = ((const uint32_t*)(tb + nf))[n];
    // ---- window + fold (:73-97)
    {
        const int mid = 3 * half;
        WARP_STRIDE(i, half) {
            const int a = mid - 1 - i, b = mid + i;
            wk[i] = -((float)tb[a] * p.win[a]) - ((float)tb[b] * p.win[b]);
            const int a2 = i, b2 = nf - 1 - i;
            wk[half + i] = ((float)tb[a2] * p.win[a2]) - ((float)tb[b2] * p.win[b2]);
        }
    }
    __syncwarp();
    // ---- DCT-IV (dct_iv.rs:49-67): pre-twiddle straight into kissfft's leaf order, levels innermost first
    WARP_STRIDE(o, N) {
        const int n = p.perm[o];
        cx[o] = cmul(ld(p.dtw, n), C2{wk[2 * n], wk[nf - 2 * n - 1]});
    }
    __syncwarp();
    for (int lv = c.n_levels - 1; lv >= 0; lv--) {
        const int pp = c.fac_p[lv], m = c.fac_m[lv], fs = c.fac_stride[lv];
        const int nbf = N / pp;
        WARP_STRIDE(b, nbf) {
            const int blk = b / m, u = b - blk * m;
            C2* f = cx + blk * (pp * m);
            switch (pp) {
                case 2: bfly2(f, p.ftw, fs, m, u); break;
                case 3: bfly3(f, p.ftw, fs, m, u); break;
                case 4: bfly4(f, p.ftw, fs, m, u); break;
                default: bfly5(f, p.ftw, fs, m, u); break;
            }
        }
        __syncwarp();
    }
    {
        const float gain = 1.0f / sqrtf(2.0f * (float)nf);
        WARP_STRIDE(n, N) {
            const C2 v = cmul(ld(p.dtw, n), cx[n]);
            const float a = v.r * 2.0f, b = -v.i * 2.0f;
            wk[2 * n] = a * gain;
            wk[nf - 2 * n - 1] = b * gain;
        }
    }
    __syncwarp();
    // ---- band energies (:140-152, divide inside the sum) and near-Nyquist flag (:154-178)
    float* e_b = p.e_b + (size_t)stream * 64;
    float* ebs = (float*)cx;                        // staging of the energies for the serial sums below
    // the terms x^2 / width of all lines in parallel (the division is the expensive part), then one ordered sum per band
    float* tq = (float*)tb;                         // the time buffer is dead by now; ne floats fit in its 2 nf int16
    WARP_STRIDE(k, ne) {
        const float width = c.band_width_of[k];                       // (band_idx[b + 1] - band_idx[b]) as f32, one load instead of three
        if (width != 0.0f) tq[k] = wk[k] * wk[k] / width;
    }
    __syncwarp();
    WARP_STRIDE(b, c.nb) {
        const int from = c.band_idx[b], to = c.band_idx[b + 1];
        float e = 0.0f;
        for (int k = from; k < to; k++) e += tq[k];
        e_b[b] = e;
        ebs[b] = e;
    }
    WARP_STRIDE(k, ne) p.xf[(size_t)stream * ne + k] = wk[k];
    __syncwarp();
    int near_nyquist = 0;
    if (c.fs <= 32000 && lane == 0) {
        const int nn_idx = c.n_ms == LC3B_7P5MS ? c.nb - 4 : c.nb - 2;
        float lo = 0.0f, hi = 0.0f;
        for (int n = 0; n < c.nb; n++) { if (n < nn_idx) lo += ebs[n]; else hi += ebs[n]; }
        near_nyquist = hi > 30.0f * lo;
    }
    if (lane == 0) p.ehand[(size_t)stream * EH_WORDS + EH_NEAR_NYQUIST] = near_nyquist;
}

// Kernel 2, one frame: attack detector and LTPF analysis of stream `stream` (per-stream state) on the input and
// hand-off record of unit `unit` (runs after enc_mdct_kernel, whose near-Nyquist flag it reads).  IDS: the CTA's warps hold
// rows stream0 .. stream0 + 3 of a subset call, whose states the shared biquad reaches through the id list; WALK: rows of
// a time-parallel call's row table.  n_live_c: warps of the CTA that have a frame now, always warps 0 .. n_live_c - 1.
template <bool IDS, bool WALK>
__device__ __forceinline__ void ltpf_frame(const AnalysisParams& p, uint8_t* smem, int stream, size_t unit, int n_live_c) {
    const EncConfig& c = *p.cfg;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int nf = c.nf;

    uint8_t* base = smem + (size_t)wid * p.smem_per_warp;
    float* wk = (float*)base;                       // 320 floats: attack scratch, later the activation sums' inputs
    float* r6 = wk + 320;                           // 98 lags
    float* rw6 = r6 + 98;                           // 98 weighted lags
    float* r12 = rw6 + 98;                          // up to 233 values
    float* x12 = r12 + 236;                         // x12_len floats
    float* x6 = x12 + c.x12_len;                    // 178 floats
    float* xs = x6 + 178;                           // x_s_ext_len (<= 540) input samples as f32 (exact)

    const int16_t* x = p.pcm + unit * p.pcm_stride;               // this frame's input samples
    int32_t* es = p.estate + (size_t)stream * ES_WORDS;
    const int near_nyquist = p.ehand[unit * EH_WORDS + EH_NEAR_NYQUIST];
    const int up = c.up, ns_keep = 240 / up;
    {   // x_s_extended (long_term_post_filter.rs:217-224): last 240/up samples of the previous frame, then this frame
        int16_t* xh = p.xs_hist + (size_t)stream * 64;
        // two samples per load (ns_keep and nf are even; the history rows are 128 bytes apart, the input row usually aligned)
        auto lo16 = [](uint32_t w) { return (float)(int16_t)(w & 0xffffu); };
        auto hi16 = [](uint32_t w) { return (float)(int16_t)(w >> 16); };
        WARP_STRIDE(n, ns_keep / 2) {
            const uint32_t w = ((const uint32_t*)xh)[n];
            xs[2 * n] = lo16(w);
            xs[2 * n + 1] = hi16(w);
        }
        if (((uintptr_t)x & 3) == 0) {
            WARP_STRIDE(n, nf / 2) {
                const uint32_t w = ((const uint32_t*)x)[n];
                xs[ns_keep + 2 * n] = lo16(w);
                xs[ns_keep + 2 * n + 1] = hi16(w);
            }
            WARP_STRIDE(n, ns_keep / 2) ((uint32_t*)xh)[n] = ((const uint32_t*)(x + nf - ns_keep))[n];
        } else {
            WARP_STRIDE(n, nf) xs[ns_keep + n] = (float)x[n];
            WARP_STRIDE(n, ns_keep) xh[n] = x[nf - ns_keep + n];
        }
    }
    __syncwarp();
    const float* xcur = xs + ns_keep;                // this frame's samples in shared memory

    // ---- attack detector (attack_detector.rs:45-105)
    int attack_detected = 0;
    {
        bool active;
        if (c.fs < 32000) active = false;
        else if (c.n_ms == LC3B_7P5MS)
            active = (c.fs == 32000 && p.nbytes >= 61 && p.nbytes < 150) || (c.fs >= 44100 && p.nbytes >= 75 && p.nbytes < 150);
        else
            active = (c.fs == 32000 && p.nbytes > 80) || (c.fs >= 41000 && p.nbytes >= 100);
        if (!active) {
            if (lane == 0) {
                es[ES_ATT_ENERGY_LAST] = (int32_t)__float_as_uint(0.0f);
                es[ES_ATT_MAX_ENERGY_LAST] = (int32_t)__float_as_uint(0.0f);
                es[ES_ATT_POS_LAST] = -1;
            }
        } else {
            int32_t* ds = (int32_t*)wk;             // num_downsampled ints, then hp floats behind them
            float* hp = wk + 160;
            const int nds = c.att_num_ds, block_len = nf / nds;
            const int tm1 = es[ES_ATT_TM1], tm2 = es[ES_ATT_TM2];
            __syncwarp();
            WARP_STRIDE(n, nds) {
                int32_t s = 0;
                for (int j = 0; j < block_len; j++) s += (int32_t)xcur[block_len * n + j];
                ds[n] = s;
            }
            __syncwarp();
            WARP_STRIDE(n, nds) {
                const float d0 = (float)ds[n];
                const float d1 = n >= 1 ? (float)ds[n - 1] : (float)tm1;
                const float d2 = n >= 2 ? (float)ds[n - 2] : (n == 1 ? (float)tm1 : (float)tm2);
                hp[n] = 0.375f * d0 - 0.5f * d1 + 0.125f * d2;
            }
            __syncwarp();
            float energy = 0.0f;
            if (lane < c.att_num_blocks)
                for (int j = 40 * lane; j < 40 * lane + 40; j++) energy += hp[j] * hp[j];
            // gather the block energies on lane 0 and run the envelope recurrence there
            float en_blk[4];
#pragma unroll
            for (int n = 0; n < 4; n++) en_blk[n] = __shfl_sync(0xffffffffu, energy, n);
            if (lane == 0) {
                float energy_last = __uint_as_float((uint32_t)es[ES_ATT_ENERGY_LAST]);
                float max_energy_last = __uint_as_float((uint32_t)es[ES_ATT_MAX_ENERGY_LAST]);
                int attack_position = -1;
                for (int n = 0; n < c.att_num_blocks; n++) {
                    const float en = en_blk[n];
                    const float a = 0.25f * max_energy_last;
                    const float max_energy = maxf_rs(a, energy_last);
                    if (en > 8.5f * max_energy) attack_position = n;
                    energy_last = en;
                    max_energy_last = max_energy;
                }
                const int pos_last = es[ES_ATT_POS_LAST];
                attack_detected = attack_position >= 0 || pos_last >= c.att_pos_limit;
                es[ES_ATT_POS_LAST] = attack_position;
                es[ES_ATT_ENERGY_LAST] = (int32_t)__float_as_uint(energy_last);
                es[ES_ATT_MAX_ENERGY_LAST] = (int32_t)__float_as_uint(max_energy_last);
                es[ES_ATT_TM1] = ds[nds - 1];
                es[ES_ATT_TM2] = ds[nds - 2];
            }
            attack_detected = __shfl_sync(0xffffffffu, attack_detected, 0);
        }
    }
    __syncwarp();

    // ---- LTPF analysis (long_term_post_filter.rs:139-215)
    constexpr int NMEM = 232, K_MIN = 17, K_MAX = 114;
    const int len12 = c.len12p8, len6 = c.len6p4;
    const int t_nbits = c.n_ms == LC3B_7P5MS ? (int)round((double)(p.nbytes * 8) * 10.0 / 7.5) : p.nbytes * 8;
    const bool gain_ltpf_on = t_nbits < 560 + c.fs_ind * 80;
    {   // shift_out_old_samples (:217-230)
        float* g12 = p.x12 + (size_t)stream * c.x12_len;
        float* g6 = p.x6 + (size_t)stream * 178;
        WARP_STRIDE(n, c.x12_len - len12) x12[n] = g12[n + len12];
        WARP_STRIDE(n, 178 - len6) x6[n] = g6[n + len6];
        WARP_STRIDE_FROM(n, 178 - len6, 178) x6[n] = 0.0f;   // overwritten below where it matters
        __syncwarp();
    }
    float* x12n = x12 + c.delay + NMEM;             // where this frame's resampled samples go
    {   // resampling (:152-166).  Output n = lane + 32 i: its phase r15 = 15 n mod up does not depend on i (up divides
        // 480), and its first input advances by 480 / up per i, so the lane's (up to four) outputs share each filter tap.
        // The reference walks k = -120/up ..= 120/up and skips taps with |up k - r15| >= 120: exactly the first one, and
        // the last one when r15 == 0 (up divides 120).  resamp_ph is the filter in phase-major order:
        // ph[j] = h[up (j - kq + 1) - r15].
        const int kq = 120 / up, q_step = 480 / up;
        const int q15 = (15 * lane) / up, r15 = (15 * lane) % up;
        const float* xp = xs + q15 + 1;
        const float* ph = c.resamp_ph + r15 * (2 * kq);
        const int n_out = len12 >> 5;                                  // 4 at 10 ms, 3 at 7.5 ms
        float a0 = 0.0f, a1 = 0.0f, a2 = 0.0f, a3 = 0.0f;
        const int last = n_out - 1;
        const float* x3 = xp + last * q_step;                          // the fourth chain repeats the last one at 7.5 ms
#pragma unroll 4
        for (int j = 0; j < 2 * kq - 1; j++) {                         // warp-uniform trip count
            const float h = ph[j];
            a0 += xp[j] * h;
            a1 += xp[q_step + j] * h;
            a2 += xp[2 * q_step + j] * h;
            a3 += x3[j] * h;
        }
        if (r15 != 0) {
            const int j = 2 * kq - 1;
            const float h = ph[j];
            a0 += xp[j] * h;
            a1 += xp[q_step + j] * h;
            a2 += xp[2 * q_step + j] * h;
            a3 += x3[j] * h;
        }
        const float sc = (float)up * c.resamp_fac;
        x12n[lane] = a0 * sc;
        x12n[lane + 32] = a1 * sc;
        x12n[lane + 64] = a2 * sc;
        if (n_out == 4) x12n[lane + 96] = a3 * sc;
    }
    // 50 Hz high-pass biquad (:169-177).  The recursive half (h50) is a serial chain: the chains of the CTA's frames run
    // side by side on the first lanes of warp 0 instead of each spending its own warp's issue slots; the feed-forward
    // half only needs h50[n], h50[n-1], h50[n-2] and runs on all lanes of the frame's own warp.
    {
        const float m1_0 = __uint_as_float((uint32_t)es[ES_H50_M1]), m2_0 = __uint_as_float((uint32_t)es[ES_H50_M2]);
        float* h50s = wk;                            // len12 <= 128 floats (attack scratch is dead by now)
        const int stream0 = blockIdx.x * ANA_WARPS;
        asm volatile("bar.sync 1, %0;" ::"r"(n_live_c * 32) : "memory");
        if (wid == 0 && lane < n_live_c) {
            uint8_t* ob = smem + (size_t)lane * p.smem_per_warp;      // warp `lane`'s slice: same carve-up as above
            float* o_wk = (float*)ob;
            const float* o_x12n = o_wk + 320 + 98 + 98 + 236 + c.delay + NMEM;
            const int o_row = WALK ? row_span(p.rows, stream0 + lane).row : state_row<IDS>(p.ids, stream0 + lane);
            int32_t* o_es = p.estate + (size_t)o_row * ES_WORDS;
            float m1 = __uint_as_float((uint32_t)o_es[ES_H50_M1]), m2 = __uint_as_float((uint32_t)o_es[ES_H50_M2]);
            for (int n = 0; n < len12; n++) {
                const float h50 = o_x12n[n] - -1.9652933726226904f * m1 - 0.9658854605688177f * m2;
                o_wk[n] = h50;
                m2 = m1;
                m1 = h50;
            }
            o_es[ES_H50_M1] = (int32_t)__float_as_uint(m1);
            o_es[ES_H50_M2] = (int32_t)__float_as_uint(m2);
        }
        asm volatile("bar.sync 1, %0;" ::"r"(n_live_c * 32) : "memory");
        WARP_STRIDE(n, len12) {
            const float h50 = h50s[n];
            const float m1 = n >= 1 ? h50s[n - 1] : m1_0;
            const float m2 = n >= 2 ? h50s[n - 2] : (n == 1 ? m1_0 : m2_0);
            x12n[n] = 0.9827947082978771f * h50 + -1.965589416595754f * m1 + 0.9827947082978771f * m2;
        }
    }
    __syncwarp();
    {   // write the shifted + new 12.8 kHz samples back (state for the next frame)
        float* g12 = p.x12 + (size_t)stream * c.x12_len;
        WARP_STRIDE(n, c.x12_len) g12[n] = x12[n];
    }
    // pitch_detection (:232-290)
    WARP_STRIDE(i, len6) {
        const float* s = x12 + NMEM - 3 + 2 * i;
        x6[K_MAX + i] = 0.1236796411180537f * s[0] + 0.2353512128364889f * s[1] + 0.2819382920909148f * s[2] +
                        0.2353512128364889f * s[3] + 0.1236796411180537f * s[4];
    }
    __syncwarp();
    {
        float* g6 = p.x6 + (size_t)stream * 178;
        WARP_STRIDE(n, 178) g6[n] = x6[n];
    }
    constexpr int NR = K_MAX + 1 - K_MIN;
    {   // 98 lags: lane l owns lags l, l+32, l+64 (and l+96 for l < 2), accumulated side by side so that the
        // x6[K_MAX + n] load and the loop are shared; each sum keeps its own order
        const int k0 = lane, k1 = lane + 32, k2 = lane + 64, k3 = lane + 96 < NR ? lane + 96 : NR - 1;
        const float* a = x6 + K_MAX;
        const float* b0 = x6 + (K_MAX - K_MIN - k0);
        const float* b1 = x6 + (K_MAX - K_MIN - k1);
        const float* b2 = x6 + (K_MAX - K_MIN - k2);
        const float* b3 = x6 + (K_MAX - K_MIN - k3);
        float s0 = 0.0f, s1 = 0.0f, s2 = 0.0f, s3 = 0.0f;
        for (int n = 0; n < len6; n++) {
            const float an = a[n];
            s0 += an * b0[n];
            s1 += an * b1[n];
            s2 += an * b2[n];
            s3 += an * b3[n];
        }
        auto put = [&](int k, float sv) {
            r6[k] = sv;
            const float weight = 1.0f - 0.5f * (float)k / (float)(K_MAX - K_MIN);
            rw6[k] = weight * sv;
        };
        put(k0, s0);
        put(k1, s1);
        put(k2, s2);
        if (lane + 96 < NR) put(k3, s3);
    }
    __syncwarp();
    int t_current = 0, pitch_present = 0;
    {
        // index_of_max (:411-423): first maximum wins; per-lane scan in ascending order, then a (value, index) reduction
        auto index_of_max_w = [&](const float* s, int n) {
            float mx = -INFINITY;
            int idx = 0x7fffffff;
            for (int i0 = 0; i0 < n; i0 += 32) {
                const int i = i0 + lane;
                if (i < n && s[i] > mx) { mx = s[i]; idx = i; }
            }
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                const float ov = __shfl_xor_sync(0xffffffffu, mx, off);
                const int oi = __shfl_xor_sync(0xffffffffu, idx, off);
                if (ov > mx || (ov == mx && oi < idx)) { mx = ov; idx = oi; }
            }
            return idx == 0x7fffffff ? 0 : idx;
        };
        const int t_prev = es[ES_T_PREV];
        const int lag_t1 = index_of_max_w(rw6, NR) + K_MIN;
        const int k_from = (K_MIN > t_prev - 4 ? K_MIN : t_prev - 4) - K_MIN;
        const int k_to = (K_MAX < t_prev + 4 ? K_MAX : t_prev + 4) - K_MIN + 1;
        const int lag_t2 = index_of_max_w(r6 + k_from, k_to - k_from) + k_from + K_MIN;
        // the three norm values are independent ordered sums of len6 terms.  Three busy lanes per warp would cost every
        // frame a warp's issue slots for the whole loop: the sums of all frames of the CTA run on the lanes of warp 0
        // (lane 3 w + j: frame of warp w, sum j), between two named barriers, like the biquad above.
        if (lane == 0) { ((int*)wk)[256] = lag_t1; ((int*)wk)[257] = lag_t2; }
        asm volatile("bar.sync 1, %0;" ::"r"(n_live_c * 32) : "memory");
        if (wid == 0 && lane < 3 * n_live_c) {
            const int w = lane / 3, j = lane - 3 * w;
            float* o_wk = (float*)(smem + (size_t)w * p.smem_per_warp);
            const float* o_x6 = o_wk + 320 + 98 + 98 + 236 + c.x12_len;
            const int lag = j == 0 ? 0 : ((const int*)o_wk)[255 + j];
            const int from = K_MAX - lag;
            float nv = 0.0f;
            for (int n = from; n < from + len6; n++) nv += o_x6[n] * o_x6[n];
            o_wk[258 + j] = nv;
        }
        asm volatile("bar.sync 1, %0;" ::"r"(n_live_c * 32) : "memory");
        const float nv0 = wk[258], nv1 = wk[259], nv2 = wk[260];
        const float normvalue1 = sqrtf(nv0 * nv1);
        const float normcorr1 = maxf_rs(0.0f, r6[lag_t1 - K_MIN] / normvalue1);
        float normcorr2;
        if (lag_t1 == lag_t2) normcorr2 = normcorr1;
        else {
            const float normvalue2 = sqrtf(nv0 * nv2);
            normcorr2 = maxf_rs(0.0f, r6[lag_t2 - K_MIN] / normvalue2);
        }
        if (normcorr2 > 0.85f * normcorr1) { t_current = lag_t2; pitch_present = normcorr2 > 0.6f; }
        else { t_current = lag_t1; pitch_present = normcorr1 > 0.6f; }
    }
    // pitch_lag_parameter (:292-363)
    const int k_min = 32 > 2 * t_current - 4 ? 32 : 2 * t_current - 4;
    const int k_max = 228 < 2 * t_current + 4 ? 228 : 2 * t_current + 4;
    const float* cur = x12 + NMEM;
    WARP_STRIDE(i, 233) r12[i] = 0.0f;
    __syncwarp();
    {                                                // at most 17 lags: one per lane
        const int k = k_min - 4 + lane;
        const int kk = k <= k_max + 4 ? k : k_max + 4;
        float cv = 0.0f;
        for (int n = 0; n < len12; n++) cv += cur[n] * cur[n - kk];
        if (k <= k_max + 4) r12[k - (k_min - 4)] = cv;
    }
    __syncwarp();
    int pitch_int = k_min, pitch_fr = 0, pitch_index = 0;
    if (lane == 0) {
        float max_corr = 0.0f;
        for (int k = k_min - 4; k <= k_max + 4; k++) {
            const float cv = r12[k - (k_min - 4)];
            if (cv > max_corr && k >= k_min && k <= k_max) { max_corr = cv; pitch_int = k; }
        }
        const int rel = pitch_int - (k_min - 4);
        auto interpolate = [&](int d) {
            float v = 0.0f;
            for (int m = -4; m <= 4; m++) {
                const int n = 4 * m - d;
                if (n > -16 && n < 16) v += r12[rel + m] * LC3T_TAB_LTPF_INTERP_R[n + 15];
            }
            return v;
        };
        if (pitch_int == 32) {
            float mx = 0.0f;
            for (int d = 0; d <= 3; d++) { const float v = interpolate(d); if (v > mx) { mx = v; pitch_fr = d; } }
        } else if (pitch_int < 127 && pitch_int > 32) {
            float mx = 0.0f;
            for (int d = -3; d <= 3; d++) { const float v = interpolate(d); if (v > mx) { mx = v; pitch_fr = d; } }
        } else if (pitch_int >= 127 && pitch_int < 157) {
            float mx = 0.0f;
            for (int d = -2; d <= 2; d += 2) { const float v = interpolate(d); if (v > mx) { mx = v; pitch_fr = d; } }
        }
        if (pitch_fr < 0) { pitch_int -= 1; pitch_fr += 4; }
        if (pitch_int < 127) pitch_index = 4 * pitch_int + pitch_fr - 128;
        else if (pitch_int < 157) pitch_index = 2 * pitch_int + pitch_fr / 2 - 126;
        else pitch_index = pitch_int + 283;
    }
    pitch_int = __shfl_sync(0xffffffffu, pitch_int, 0);
    pitch_fr = __shfl_sync(0xffffffffu, pitch_fr, 0);
    pitch_index = __shfl_sync(0xffffffffu, pitch_index, 0);
    // activation_bit (:365-409): per-sample interpolated values in parallel, the three running sums serially
    float* nd_a = wk;                                // len12 floats each (2 * 128 <= nf for every config? no: checked below)
    float* sh_a = wk + 128;
    auto dot = [&](int n, int d) {
        float v = 0.0f;
        for (int k = -2; k <= 2; k++) {
            const int hi = 4 * k - d;
            if (hi > -8 && hi < 8) v += x12[NMEM + n - k] * LC3T_TAB_LTPF_INTERP_X12K8[hi + 7];
        }
        return v;
    };
    __syncwarp();
    WARP_STRIDE(n, len12) {
        nd_a[n] = dot(n, 0);
        sh_a[n] = dot(n - pitch_int, pitch_fr);
    }
    __syncwarp();
    // the three running sums (nd*sh, nd*nd, sh*sh) are independent ordered sums of len12 terms: again on warp 0 for all
    // frames of the CTA (lane 3 w + j)
    asm volatile("bar.sync 1, %0;" ::"r"(n_live_c * 32) : "memory");
    if (wid == 0 && lane < 3 * n_live_c) {
        const int w = lane / 3, j = lane - 3 * w;
        float* o_wk = (float*)(smem + (size_t)w * p.smem_per_warp);
        const float* o_nd = o_wk;
        const float* o_sh = o_wk + 128;
        const float* pa = j == 2 ? o_sh : o_nd;
        const float* pb = j == 1 ? o_nd : o_sh;
        float acc = 0.0f;
        for (int n = 0; n < len12; n++) acc += pa[n] * pb[n];
        o_wk[258 + j] = acc;
    }
    asm volatile("bar.sync 1, %0;" ::"r"(n_live_c * 32) : "memory");
    const float acc3 = wk[258], nd_tot = wk[259], sh_tot = wk[260];
    if (lane == 0) {
        const float nc_num = acc3;
        const float nc_den = sqrtf(nd_tot * sh_tot);
        float nc = nc_den > 0.0f ? nc_num / nc_den : 0.0f;
        const float pitch = (float)pitch_int + (float)pitch_fr / 4.0f;
        const bool mem_active = es[ES_MEM_LTPF_ACTIVE] != 0;
        const float mem_nc = __uint_as_float((uint32_t)es[ES_MEM_NC]);
        const float mem_mem_nc = __uint_as_float((uint32_t)es[ES_MEM_MEM_NC]);
        const float mem_pitch = __uint_as_float((uint32_t)es[ES_MEM_PITCH]);
        bool ltpf_active = false;
        if (gain_ltpf_on && !near_nyquist) {
            ltpf_active = (!mem_active && (c.n_ms == LC3B_10MS || mem_mem_nc > 0.94f) && mem_nc > 0.94f && nc > 0.94f) ||
                          (mem_active && nc > 0.9f) ||
                          (mem_active && fabsf(pitch - mem_pitch) < 2.0f && (nc - mem_nc) > -0.1f && nc > 0.84f);
        }
        if (!pitch_present) { pitch_index = 0; nc = 0.0f; }
        es[ES_T_PREV] = t_current;
        es[ES_MEM_MEM_NC] = (int32_t)__float_as_uint(mem_nc);
        if (pitch_present) {
            es[ES_MEM_PITCH] = (int32_t)__float_as_uint(pitch);
            es[ES_MEM_LTPF_ACTIVE] = ltpf_active;
            es[ES_MEM_NC] = (int32_t)__float_as_uint(nc);
        } else {
            es[ES_MEM_PITCH] = (int32_t)__float_as_uint(0.0f);
            es[ES_MEM_LTPF_ACTIVE] = 0;
            es[ES_MEM_NC] = (int32_t)__float_as_uint(0.0f);
        }
        int32_t* eh = p.ehand + unit * EH_WORDS;
        eh[EH_ATTACK] = attack_detected;
        eh[EH_PITCH_INDEX] = pitch_index;
        eh[EH_PITCH_PRESENT] = pitch_present;
        eh[EH_LTPF_ACTIVE] = ltpf_active;
        eh[EH_NBITS_LTPF] = pitch_present ? 11 : 1;
    }
}

// Kernel 2: one frame per warp (lc3b_encode_frames; IDS: lc3b_encode_frames_subset), or, WALK (always with IDS: a row's
// state row comes from the row table), a warp per row of a time-parallel call's row table walking the row's frames in
// order.  The walk is a separate instantiation, so the frame-by-frame path keeps its registers.  The __syncwarp orders
// the state lane 0 (and warp 0, for the biquad) wrote in frame f before the lanes read it in frame f + 1.  The table is
// sorted by count, descending, so the warps of a CTA that still have frame f are warps 0 .. n_live - 1, n_live the number
// of the CTA's rows with count > f: the named barriers count exactly them, a warp leaves when its row is done, and warp 0
// (the CTA's longest row) is there for every frame to do the ordered sums of lanes < n_live.
template <bool WALK, bool IDS>
__global__ void __launch_bounds__(ANA_WARPS * 32) enc_ltpf_kernel(AnalysisParams p) {
    static_assert(!WALK || IDS, "the row walk addresses state through the row table");
    extern __shared__ __align__(16) uint8_t smem[];
    const int stream = blockIdx.x * ANA_WARPS + (threadIdx.x >> 5);
    if (stream >= p.n_streams) return;
    const int n_cta = min(ANA_WARPS, p.n_streams - (int)blockIdx.x * ANA_WARPS);   // the CTA's rows
    if constexpr (WALK) {
        const int lane = threadIdx.x & 31;
        const RowSpan rs = row_span(p.rows, stream);
        const int cnt = lane < n_cta ? row_span(p.rows, blockIdx.x * ANA_WARPS + lane).count : 0;   // lane j: warp j's
        // the count and the live warps as warp reductions: their results are uniform registers, so the walk's control flow
        // stays on the uniform datapath (as with a frame count in a kernel parameter; as per-lane values it ran 4-5 % slower)
        const int F = __reduce_max_sync(0xffffffffu, rs.count);
        for (int f = 0; f < F; f++) {
            ltpf_frame<true, true>(p, smem, rs.row, (size_t)rs.off + f, __reduce_add_sync(0xffffffffu, cnt > f ? 1u : 0u));
            __syncwarp();
        }
    } else {
        ltpf_frame<IDS, false>(p, smem, state_row<IDS>(p.ids, stream), (size_t)stream, n_cta);
    }
}

static size_t mdct_warp_bytes(int nf) {
    size_t per_warp = (size_t)nf * 4 + (size_t)(nf / 2) * 8 + (size_t)2 * nf * 2;
    return (per_warp + 15) & ~(size_t)15;
}
static size_t ltpf_warp_bytes(const lc3b_config& c) {
    const int x12_len = (c.n_ms == LC3B_10MS ? 128 + 24 : 96 + 44) + 232;
    // 320 scratch floats (160 + 160 attack scratch, 2 x 128 activation scratch), 98 + 98 + 236 correlation values,
    // the 12.8 kHz and 6.4 kHz buffers, the input samples as f32
    size_t per_warp = (size_t)(320 + 98 + 98 + 236 + x12_len + 178 + 544) * 4;
    return (per_warp + 15) & ~(size_t)15;
}

// dynamic shared memory limits, once per handle (lc3b_encoder_init)
cudaError_t prepare_enc_analysis(const EncoderState& st) {
    const int mb = (int)(mdct_warp_bytes(st.cfg.nf) * ANA_WARPS), lb = (int)(ltpf_warp_bytes(st.cfg) * ANA_WARPS);
    cudaError_t e = cudaFuncSetAttribute(enc_mdct_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, mb);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(enc_mdct_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, mb);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(enc_ltpf_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, lb);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(enc_ltpf_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, lb);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(enc_ltpf_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, lb);
    return e;
}

void plan_enc_analysis(LaunchPlan& plan, const EncoderState& st, const int16_t* pcm, size_t pcm_stride, int nbytes, int stages,
                       const int32_t* ids, const int32_t* rows, int n_rows) {
    AnalysisParams p;
    memset(&p, 0, sizeof(p));
    p.cfg = st.ecfg;
    p.win = st.win;
    p.dtw = st.dtw;
    p.ftw = st.ftw;
    p.perm = st.perm;
    p.pcm = pcm;
    p.pcm_stride = pcm_stride;
    p.nbytes = nbytes;
    p.n_streams = st.n_streams;
    p.thist = st.thist;
    p.xs_hist = st.xs_hist;
    p.x12 = st.x12;
    p.x6 = st.x6;
    p.estate = st.estate;
    p.xf = st.xf;
    p.e_b = st.e_b;
    p.ehand = st.ehand;
    p.ids = ids;
    p.rows = rows;
    if (stages & 1) {
        const size_t per_warp = mdct_warp_bytes(st.cfg.nf);
        p.smem_per_warp = (int)per_warp;
        plan.add(ids ? enc_mdct_kernel<true> : enc_mdct_kernel<false>, (unsigned)((st.n_streams + ANA_WARPS - 1) / ANA_WARPS),
                 ANA_WARPS * 32, per_warp * ANA_WARPS, p);
    }
    if (stages & 2) {
        const size_t per_warp = ltpf_warp_bytes(st.cfg);
        p.smem_per_warp = (int)per_warp;
        if (rows) p.n_streams = n_rows;                         // one warp per row, walking its frames
        plan.add(rows ? enc_ltpf_kernel<true, true> : ids ? enc_ltpf_kernel<false, true> : enc_ltpf_kernel<false, false>,
                 (unsigned)((p.n_streams + ANA_WARPS - 1) / ANA_WARPS), ANA_WARPS * 32, per_warp * ANA_WARPS, p);
    }
}

}  // namespace lc3b
