// lc3b engine: the synthesis pieces that both decode paths run around the inverse MDCT (lc3b_imdct.cuh): concealment,
// long-term post filter and PCM rounding.  The frame-by-frame kernels (lc3b_dec_synth.cu) and the time-parallel ones
// (lc3b_dec_multi.cu) promise identical bits, so each piece is written once, here.
//
//   PacketLossConcealment::load_into          src/decoder/packet_loss_concealment.rs:63-85
//   LongTermPostFilter::run                   src/decoder/long_term_post_filter.rs:142-424
//   output_scaling::scale_and_round           src/decoder/output_scaling.rs:13-26
//
// Every f32 operation is an explicit xa/xs/xm/xd intrinsic, in the reference's order.
#pragma once
#include <stdint.h>

#include "lc3b_common.cuh"
#include "lc3b_math.cuh"

namespace lc3b {

__device__ __forceinline__ int32_t round_pcm_i32(float v) {          // output_scaling.rs:13-26
    int32_t q = v > 0.0f ? cast_i32(xa(v, 0.5f)) : cast_i32(xs(v, 0.5f));
    return q > 32767 ? 32767 : q < -32768 ? -32768 : q;
}

// ---------------------------------------------------------------- concealment (packet_loss_concealment.rs:63-85)
__device__ __forceinline__ uint32_t plc_lcg(uint32_t s) { return (16831u + s * 12821u) & 0xFFFFu; }

// n steps of plc_lcg composed into one: s_n = (a * s_0 + c) & 0xFFFF
struct PlcJump {
    uint32_t a, c;
    __device__ __forceinline__ uint32_t step(uint32_t s) const { return (a * s + c) & 0xFFFFu; }
};
__device__ __forceinline__ PlcJump plc_lcg_jump(int n) {
    PlcJump j{1, 0};
    for (int i = 0; i < n; i++) { j.c = plc_lcg(j.c); j.a = (j.a * 12821u) & 0xFFFFu; }
    return j;
}

// the fade of a concealed frame: alpha as it enters the frame after `lost` lost frames
__device__ __forceinline__ float plc_fade(float alpha, int lost) { return lost >= 4 ? xm(alpha, lost < 8 ? 0.9f : 0.85f) : alpha; }

// One warp fills P[0 .. NF) with the concealed spectrum: line k < NE is src[k] * (+-alpha), its sign from the LCG advanced
// k + 1 times from `seed`; lines from NE on are zero.  A lane's first line is k = lane, then it jumps 32 lines at a time.
// seed_out, if given, receives the LCG state after the NE lines (the seed of the next concealed frame).  src may be P.
template <int NF, int NE>
__device__ __forceinline__ void plc_scramble(float* P, const float* src, float alpha, uint32_t seed, int lane,
                                             int32_t* seed_out = nullptr) {
    uint32_t s = seed;
    for (int i = 0; i <= lane; i++) s = plc_lcg(s);
    const PlcJump j32 = plc_lcg_jump(32);
    // walking pointers rather than P[k] / src[k]: inlined into synth_classic_kernel, this form keeps its register count
    float* dst = P + lane;
    const float* in = src + lane;
    for (int k = lane; k < NF; k += 32, dst += 32, in += 32) {
        float v = 0.0f;
        if (k < NE) {
            const float lg = *in;
            v = s < 0x8000u ? xm(lg, alpha) : xm(lg, -alpha);
            if (seed_out && k == NE - 1) *seed_out = (int32_t)s;
            s = j32.step(s);
        }
        *dst = v;
    }
}

// ---------------------------------------------------------------- long-term post filter
// One frame's filter parameters.  code: gain-table row 0..3, 4 = zero gains.  The default is the filter switched off.
struct LtpfPar { int active = 0, p_int = 0, p_fr = 0, code = 4; };

// compute_filter_parameters :164-190 and compute_gains_params :142-161, from the frame's side record
__device__ __forceinline__ LtpfPar ltpf_params(const DevConfig& c, const int32_t* sd) {
    LtpfPar r;
    r.active = sd[SD_LTPF_ACTIVE];
    if (r.active) {
        const int pi = sd[SD_PITCH_INDEX], nbits = sd[SD_NBITS];
        int pit;
        double pfr;
        if (pi >= 440) { pit = pi - 283; pfr = 0.0; }
        else if (pi >= 380) { pit = pi / 2 - 63; pfr = (double)(2 * pi - 4 * pit - 252); }
        else { pit = pi / 4 + 32; pfr = (double)(pi + 128 - 4 * pit); }
        const double pitch = (double)pit + pfr / 4.0;
        const double pitch_fs = pitch * (8000.0 * ceil((double)c.fs / 8000.0) / 12800.0);
        const int p_up = (int)((pitch_fs * 4.0) + 0.5);
        r.p_int = p_up / 4;
        r.p_fr = p_up - 4 * r.p_int;
        const int t_nbits = c.n_ms == LC3B_7P5MS ? (int)round((double)nbits * 10.0 / 7.5) : nbits;
        const int sf = c.fs_ind * 80;
        r.code = t_nbits < 320 + sf ? 0 : t_nbits < 400 + sf ? 1 : t_nbits < 480 + sf ? 2 : t_nbits < 560 + sf ? 3 : 4;
    }
    return r;
}

// The previous frame's parameters in the per-stream state: SS_LTPF_PREV (bit 0 = active, bits 8.. = code),
// SS_LTPF_PINT and SS_LTPF_PFR.
__device__ __forceinline__ int ltpf_prev_active(int32_t prev_word) { return prev_word & 1; }
__device__ __forceinline__ LtpfPar ltpf_load_prev(const int32_t* ss) {
    const int32_t w = ss[SS_LTPF_PREV];
    LtpfPar r;
    r.active = ltpf_prev_active(w);
    r.p_int = ss[SS_LTPF_PINT];
    r.p_fr = ss[SS_LTPF_PFR];
    r.code = w >> 8;
    return r;
}
__device__ __forceinline__ void ltpf_store_prev(int32_t* ss, const LtpfPar& q) {
    ss[SS_LTPF_PREV] = (q.active ? 1 : 0) | (q.code << 8);
    ss[SS_LTPF_PINT] = q.p_int;
    ss[SS_LTPF_PFR] = q.p_fr;
}

// Per-warp shared-memory buffer of the post-filter kernels, in this order:
//   Y        blocks * nf floats   the circular output history x_hat_ltpf_mem (long_term_post_filter.rs:30)
//   X        nf                   this frame's x_hat, the filter input
//   xt       16                   the last 16 samples of the previous frame's x_hat
//   scratch  l_num + norm         frozen history for transition case 5
static inline size_t ltpf_warp_bytes(const lc3b_config& c) {
    const int blocks = c.n_ms == LC3B_10MS ? 2 : 3;
    size_t b = (size_t)(blocks * c.nf + c.nf + 16 + 16 + c.nf / 3 + 16) * 4;
    return (b + 15) & ~(size_t)15;
}

// The configuration's filter sizes, hist_len = blocks * nf floats of ring.  A kernel reads them once, before its loop over
// streams or frames, and passes the ring length it has as a kernel parameter: read again for every frame (past the
// loop's global stores) or kept as a product of its own, they cost ltpf_multi_kernel registers and spills.
struct LtpfGeo { int nf, blocks, hist_len, l_num, l_den, norm, s2p5; };
__device__ __forceinline__ LtpfGeo ltpf_geo(const DevConfig& c, int hist_len) {
    return {c.nf, c.ltpf_blocks, hist_len, c.ltpf_l_num, c.ltpf_l_den, c.ltpf_norm, c.ltpf_s2p5};
}

// long_term_post_filter.rs:252-424, all five transition cases: one warp writes Y[blk .. blk + nf) from X, xt and the
// history in Y, with cur / prev the parameters of this frame and of the previous one.  The recursion reaches back at
// least p_int - l_den/2 >= 18 samples, so up to 32 consecutive outputs are computed in parallel per step.
__device__ __forceinline__ void ltpf_filter_frame(const DevConfig& c, const LtpfGeo& g, float* Y, const float* X, const float* xt,
                                                  float* scratch, int blk, const LtpfPar& cur, const LtpfPar& prev, int lane) {
    const int nf = g.nf, blocks = g.blocks, hist_len = g.hist_len, l_num = g.l_num, l_den = g.l_den, norm = g.norm, s2p5 = g.s2p5;
    // coefficient sets: current (c_num, c_den) and previous (c_num_mem, c_den_mem); code 4 = all zero
    auto cnum = [&](int cd, int k) -> float { return cd < 4 ? c.ltpf_num[cd][k] : 0.0f; };
    auto cden = [&](int cd, int fr, int k) -> float { return cd < 4 ? c.ltpf_den[cd][fr][k] : 0.0f; };
    const int cur_code = cur.active ? cur.code : 4;     // inactive: zeroed coefficients (:196-201)
    const int mem_code = prev.active ? prev.code : 4;
    auto wrapi = [&](int idx) -> int { return idx < 0 ? idx + hist_len : idx; };   // :244-250
    auto x_at = [&](int pos) -> float {                 // x_hat_mem[wrap(pos)], pos relative to buffer start
        const int rel = pos - blk;                      // >= -l_num
        return rel >= 0 ? X[rel] : xt[16 + rel];
    };
    // compute_filter / compute_filter_mem :380-415
    auto filt = [&](int start, int pint, int cd, int fr) -> float {
        float out = 0.0f;
        for (int k = 0; k <= l_num; k++) out = xa(out, xm(cnum(cd, k), x_at(start - k)));
        const int sden = start - pint + l_den / 2;
        for (int k = 0; k <= l_den; k++) out = xs(out, xm(cden(cd, fr, k), Y[wrapi(sden - k)]));
        return out;
    };
    const float fnorm = (float)norm;
    // run `body(n)` for n in [n0, n1) in dependency-safe chunks: outputs reach back at least `reach` samples
    auto chunked = [&](int n0, int n1, int reach, auto body) {
        const int C = reach < 32 ? reach : 32;
        for (int s = n0; s < n1; s += C) {
            const int n = s + lane;
            if (lane < C && n < n1) body(n);
            __syncwarp();
        }
    };
    const int reach_cur = cur.active ? cur.p_int - l_den / 2 : 32;
    const int reach_mem = prev.active ? prev.p_int - l_den / 2 : 32;
    auto deactivate_first = [&]() {                     // :417-424
        chunked(0, s2p5, reach_mem, [&](int n) {
            float fo = filt(blk + n, prev.p_int, mem_code, prev.p_fr);
            fo = xm(fo, xs(1.0f, xd((float)n, fnorm)));
            Y[blk + n] = xs(X[n], fo);
        });
    };
    auto plain_from = [&](int n0) {
        chunked(n0, nf, reach_cur, [&](int n) { Y[blk + n] = xs(X[n], filt(blk + n, cur.p_int, cur_code, cur.p_fr)); });
    };
    if (cur.active && !prev.active) {                   // case 2
        chunked(0, s2p5, reach_cur, [&](int n) {
            float fo = filt(blk + n, cur.p_int, cur_code, cur.p_fr);
            fo = xm(fo, xd((float)n, fnorm));
            Y[blk + n] = xs(X[n], fo);
        });
        plain_from(s2p5);
    } else if (!cur.active && prev.active) {            // case 3
        deactivate_first();
        for (int n = s2p5 + lane; n < nf; n += 32) Y[blk + n] = X[n];
    } else if (cur.p_int == prev.p_int && cur.p_fr == prev.p_fr) {   // case 4
        plain_from(0);
    } else {                                            // case 5
        deactivate_first();
        // activate_first_2p5ms_from_mem :345-378: numerator taps read a frozen copy of y[blk-l_num .. blk+norm)
        for (int i = lane; i < l_num + norm; i += 32) {
            int src;
            if (blk < l_num) src = i < l_num ? blocks * nf - l_num + i : i - l_num;
            else src = blk - l_num + i;
            scratch[i] = Y[src];
        }
        __syncwarp();
        chunked(0, s2p5, reach_cur, [&](int n) {
            float fo = 0.0f;
            for (int k = 0; k <= l_num; k++) fo = xa(fo, xm(cnum(cur_code, k), scratch[l_num + n - k]));
            const int sden = blk + n - cur.p_int + l_den / 2;
            for (int k = 0; k <= l_den; k++) fo = xs(fo, xm(cden(cur_code, cur.p_fr, k), Y[wrapi(sden - k)]));
            fo = xm(fo, xd((float)n, fnorm));
            Y[blk + n] = xs(scratch[n + l_num], fo);
        });
        plain_from(s2p5);
    }
    __syncwarp();
}

}  // namespace lc3b
