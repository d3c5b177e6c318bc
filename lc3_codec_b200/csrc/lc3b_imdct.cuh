// lc3b engine: low-delay inverse MDCT of one frame by one warp, frame length known at compile time.
//
//   ModDiscreteCosTrans::run / apply_mdct_inverse   src/decoder/modified_dct.rs:76-136
//   DiscreteCosTransformIv::run                     src/common/dct_iv.rs:49-67
//   KissFastFourierTransform::transform             src/common/kissfft.rs:78 (replaced: see below)
//
// The DCT-IV is pre-twiddle + N = nf/2 point complex FFT + post-twiddle.  The FFT is a shared-memory Stockham
// autosort with radix-5/3/4/2 stages whose sizes, strides and trip counts are template constants, so every stage
// is straight-line code: the pre-twiddle is folded into the first stage (which needs no FFT twiddles) and the
// post-twiddle into the last.  It uses another factor order than kissfft: the PCM contract is +-1 LSB, not bit
// equality.  All products are written with explicit fma/mul intrinsics so that the frame-by-frame kernel and the
// time-parallel kernel, which both instantiate this header, produce identical bits.  dct_iv_pair computes the same
// butterflies for two frames per warp with all stages in registers and one shared-memory exchange (bit-identical too).
//
// The unfolded, windowed 2*nf samples leave in registers, two consecutive samples per lane and step:
//   head[n] = t[z + n]      * w[z + n]        n in [0, nf)      (added to the overlap memory / output)
//   tail[n] = t[nf + z + n] * w[nf + z + n]   n in [0, nf - z)  (next frame's overlap memory)
// with element (j, e) of a lane being n = 64 * j + 2 * lane + e.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace lc3b {

template <int NF, bool MS10>
struct FrameGeo {
    static constexpr int N = NF / 2;                                    // FFT length
    static constexpr int Z = MS10 ? 3 * NF / 8 : 7 * NF / 30;           // common/config.rs:42-100
    static constexpr int NE = MS10 ? (NF < 400 ? NF : 400) : (NF < 300 ? NF : 300);
    static constexpr int NP = (NF + 63) / 64;                           // lane steps covering nf samples in pairs
    static constexpr int NPT = (NF - Z + 63) / 64;                      // ... covering the nf - z overlap samples
};

// Stockham stage radices per FFT length: the 5 first (the first stage has no twiddles), then 3s, 4s, 2
template <int N> struct FftPlan;
template <> struct FftPlan<30>  { static constexpr int n = 3; static constexpr int r(int i) { constexpr int v[4] = {5, 3, 2, 0}; return v[i]; } };
template <> struct FftPlan<40>  { static constexpr int n = 3; static constexpr int r(int i) { constexpr int v[4] = {5, 4, 2, 0}; return v[i]; } };
template <> struct FftPlan<60>  { static constexpr int n = 3; static constexpr int r(int i) { constexpr int v[4] = {5, 3, 4, 0}; return v[i]; } };
template <> struct FftPlan<80>  { static constexpr int n = 3; static constexpr int r(int i) { constexpr int v[4] = {5, 4, 4, 0}; return v[i]; } };
template <> struct FftPlan<90>  { static constexpr int n = 4; static constexpr int r(int i) { constexpr int v[4] = {5, 3, 3, 2}; return v[i]; } };
template <> struct FftPlan<120> { static constexpr int n = 4; static constexpr int r(int i) { constexpr int v[4] = {5, 3, 4, 2}; return v[i]; } };
template <> struct FftPlan<160> { static constexpr int n = 4; static constexpr int r(int i) { constexpr int v[4] = {5, 4, 4, 2}; return v[i]; } };
template <> struct FftPlan<180> { static constexpr int n = 4; static constexpr int r(int i) { constexpr int v[4] = {5, 3, 3, 4}; return v[i]; } };
template <> struct FftPlan<240> { static constexpr int n = 4; static constexpr int r(int i) { constexpr int v[4] = {5, 3, 4, 4}; return v[i]; } };

namespace imdct_detail {

__device__ __forceinline__ float2 cmul(float2 a, float2 b) {
    return make_float2(__fmaf_rn(a.x, b.x, -__fmul_rn(a.y, b.y)), __fmaf_rn(a.x, b.y, __fmul_rn(a.y, b.x)));
}
__device__ __forceinline__ float2 cadd(float2 a, float2 b) { return make_float2(__fadd_rn(a.x, b.x), __fadd_rn(a.y, b.y)); }
__device__ __forceinline__ float2 csub(float2 a, float2 b) { return make_float2(__fsub_rn(a.x, b.x), __fsub_rn(a.y, b.y)); }

template <int R> __device__ __forceinline__ void dft(float2 (&v)[R]);
template <> __device__ __forceinline__ void dft<2>(float2 (&v)[2]) {
    const float2 a = v[0], b = v[1];
    v[0] = cadd(a, b);
    v[1] = csub(a, b);
}
template <> __device__ __forceinline__ void dft<3>(float2 (&v)[3]) {
    const float S = 0.86602540378443864676f;                            // sin(2 pi / 3)
    const float2 t = cadd(v[1], v[2]), d = csub(v[1], v[2]);
    const float2 m = make_float2(__fmaf_rn(-0.5f, t.x, v[0].x), __fmaf_rn(-0.5f, t.y, v[0].y));
    const float2 r = make_float2(__fmul_rn(S, d.y), -__fmul_rn(S, d.x));   // -i * sin * d  (forward transform)
    v[0] = cadd(v[0], t);
    v[1] = cadd(m, r);
    v[2] = csub(m, r);
}
template <> __device__ __forceinline__ void dft<4>(float2 (&v)[4]) {
    const float2 a = cadd(v[0], v[2]), b = csub(v[0], v[2]);
    const float2 c = cadd(v[1], v[3]), d = csub(v[1], v[3]);
    const float2 dj = make_float2(d.y, -d.x);                           // -i * d
    v[0] = cadd(a, c);
    v[1] = cadd(b, dj);
    v[2] = csub(a, c);
    v[3] = csub(b, dj);
}
template <> __device__ __forceinline__ void dft<5>(float2 (&v)[5]) {
    const float C1 = 0.30901699437494742410f, C2 = -0.80901699437494742410f;   // cos(2pi/5), cos(4pi/5)
    const float S1 = 0.95105651629515357212f, S2 = 0.58778525229247312917f;    // sin(2pi/5), sin(4pi/5)
    const float2 a1 = cadd(v[1], v[4]), b1 = csub(v[1], v[4]);
    const float2 a2 = cadd(v[2], v[3]), b2 = csub(v[2], v[3]);
    const float2 m1 = make_float2(__fmaf_rn(C2, a2.x, __fmaf_rn(C1, a1.x, v[0].x)), __fmaf_rn(C2, a2.y, __fmaf_rn(C1, a1.y, v[0].y)));
    const float2 m2 = make_float2(__fmaf_rn(C1, a2.x, __fmaf_rn(C2, a1.x, v[0].x)), __fmaf_rn(C1, a2.y, __fmaf_rn(C2, a1.y, v[0].y)));
    // forward transform: X[k] = m - i * (S..) * b ;  -i * (x + iy) = (y, -x)
    const float2 n1 = make_float2(__fmaf_rn(S2, b2.y, __fmul_rn(S1, b1.y)), -__fmaf_rn(S2, b2.x, __fmul_rn(S1, b1.x)));
    const float2 n2 = make_float2(__fmaf_rn(-S1, b2.y, __fmul_rn(S2, b1.y)), -__fmaf_rn(-S1, b2.x, __fmul_rn(S2, b1.x)));
    v[0] = make_float2(__fadd_rn(__fadd_rn(v[0].x, a1.x), a2.x), __fadd_rn(__fadd_rn(v[0].y, a1.y), a2.y));
    v[1] = cadd(m1, n1);
    v[4] = csub(m1, n1);
    v[2] = cadd(m2, n2);
    v[3] = csub(m2, n2);
}

// One Stockham stage over the warp.  FIRST: the input is the real spectrum `xr` (nf floats) and the DCT-IV
// pre-twiddle z[n] = dtw[n] * (x[2n] + i x[nf-1-2n]) is applied on the fly.  LAST: the DCT-IV post-twiddle is
// applied and the result is scattered as nf real coefficients into `yr`.
template <int NF, int R, int NS, bool FIRST, bool LAST>
__device__ __forceinline__ void stage(const float* __restrict__ xr, const float2* __restrict__ xc, float2* __restrict__ yc,
                                      float* __restrict__ yr, const float2* __restrict__ dtw, const float2* __restrict__ ftw,
                                      int lane) {
    constexpr int N = NF / 2, NBF = N / R, TW = N / (NS * R);
#pragma unroll
    for (int j0 = 0; j0 < NBF; j0 += 32) {
        const int j = j0 + lane;
        if (j0 + 32 <= NBF || j < NBF) {
            const int k = j % NS;
            float2 v[R];
#pragma unroll
            for (int t = 0; t < R; t++) {
                const int n = j + t * NBF;
                if (FIRST) v[t] = cmul(dtw[n], make_float2(xr[2 * n], xr[NF - 1 - 2 * n]));
                else {
                    v[t] = xc[n];
                    if (t > 0 && NS > 1) v[t] = cmul(v[t], ftw[k * t * TW]);
                }
            }
            dft<R>(v);
            const int base = (j - k) * R + k;
#pragma unroll
            for (int t = 0; t < R; t++) {
                const int o = base + t * NS;
                if (LAST) {
                    const float2 w = cmul(dtw[o], v[t]);
                    yr[2 * o] = __fmul_rn(w.x, 2.0f);
                    yr[NF - 1 - 2 * o] = __fmul_rn(w.y, -2.0f);
                } else yc[o] = v[t];
            }
        }
    }
}

template <int NF, int S, int NS>
__device__ __forceinline__ void stages(float* P, float* Q, const float2* __restrict__ dtw, const float2* __restrict__ ftw, int lane) {
    using Plan = FftPlan<NF / 2>;
    if constexpr (S < Plan::n) {
        constexpr int R = Plan::r(S);
        constexpr bool first = S == 0, last = S == Plan::n - 1;
        float* src = (S & 1) ? Q : P;                                   // stage s reads P, Q, P, Q ... and writes the other
        float* dst = (S & 1) ? P : Q;
        stage<NF, R, NS, first, last>(src, (const float2*)src, (float2*)dst, dst, dtw, ftw, lane);
        __syncwarp();
        stages<NF, S + 1, NS * R>(P, Q, dtw, ftw, lane);
    }
}

// ---- The same FFT with every stage in registers but one exchange through shared memory (dct_iv_pair below).
// With G = r0 * r1 and L = N / G, the Stockham index maps of stage<> split into two register-resident halves:
//  * pass A, stages 0 and 1, lane a < L: stage 1's butterflies j = r0 * a + k (k < r0) read the outputs of stage 0's
//    butterflies a + L * t (t < r1), so the lane runs those r1 butterflies, then the r0 butterflies of stage 1 on the
//    values it holds; its G outputs are the contiguous positions G * a ... G * a + G - 1;
//  * pass B, stages 2 .. n - 1, lane k < G: every later stage reads and writes only positions = k (mod G) (all its
//    strides and butterfly counts are multiples of G), so the lane gathers "column" k (positions G * m + k, m < L) and
//    runs the remaining stages on it as a Stockham FFT of L points whose twiddle index carries the column.
// Every butterfly sees the inputs, twiddle and dft<R> / cmul sequence of stage<>: the output is bit-identical.
template <int N>
struct RegFftPlan {
    using Plan = FftPlan<N>;
    static constexpr int R0 = Plan::r(0), R1 = Plan::r(1), G = R0 * R1, L = N / G;
    static constexpr bool half_warp = Plan::n >= 3 && G <= 16 && L <= 16;   // one frame fits half a warp in both passes
};

// Pass B from stage S on: x[m] is position G * m + k, NSM = (stage S's NS) / G.  The last stage applies the DCT-IV
// post-twiddle and scatters into yr.  `odd` (the warp's second frame) swaps the order of the two scatter stores, so
// that one store instruction writes even words for one frame and odd words for the other: no bank conflicts.
template <int NF, int S, int NSM>
__device__ __forceinline__ void column_stages(const float2 (&x)[RegFftPlan<NF / 2>::L], float* __restrict__ yr, const float2* __restrict__ dtw,
                                              const float2* __restrict__ ftw, int k, bool odd) {
    using Plan = FftPlan<NF / 2>;
    constexpr int N = NF / 2, G = RegFftPlan<N>::G, L = RegFftPlan<N>::L, R = Plan::r(S), NBF = L / R, TW = N / (G * NSM * R);
    constexpr bool last = S == Plan::n - 1;
    float2 y[L];
#pragma unroll
    for (int jm = 0; jm < NBF; jm++) {
        const int km = jm % NSM;
        float2 v[R];
#pragma unroll
        for (int t = 0; t < R; t++) {
            v[t] = x[jm + t * NBF];
            if (t > 0) v[t] = cmul(v[t], ftw[(G * km + k) * t * TW]);
        }
        dft<R>(v);
#pragma unroll
        for (int t = 0; t < R; t++) {
            const int m = (jm - km) * R + km + t * NSM;
            if constexpr (last) {
                const int o = G * m + k;
                const float2 w = cmul(dtw[o], v[t]);
                const float re = __fmul_rn(w.x, 2.0f), im = __fmul_rn(w.y, -2.0f);
                yr[odd ? NF - 1 - 2 * o : 2 * o] = odd ? im : re;
                yr[odd ? 2 * o : NF - 1 - 2 * o] = odd ? re : im;
            } else y[m] = v[t];
        }
    }
    if constexpr (!last) column_stages<NF, S + 1, NSM * R>(y, yr, dtw, ftw, k, odd);
}

}  // namespace imdct_detail

// DCT-IV of the nf floats in P (spectrum, zero padded beyond ne); P and Q are nf floats each (8-byte aligned).
// Returns the buffer that holds the nf output coefficients.
template <int NF>
__device__ __forceinline__ float* dct_iv_warp(float* P, float* Q, const float2* __restrict__ dtw, const float2* __restrict__ ftw, int lane) {
    imdct_detail::stages<NF, 0, 1>(P, Q, dtw, ftw, lane);
    return (FftPlan<NF / 2>::n & 1) ? Q : P;
}

// DCT-IV of two frames per warp, one per half warp, bit-identical to dct_iv_warp: passes A and B above with a single
// exchange through X in between.  Per half: P = the frame's nf floats (spectrum in, the nf output coefficients out, in
// place), X = nf floats of exchange space, l = lane within the half, odd = second half, live = the half has a frame.
// Every lane of the warp must call it (it synchronises the warp).  Per frame and pass A lane: 2 G shared loads, G
// pre-twiddle loads, one shared store per position; per pass B lane: L shared loads, L post-twiddle loads, 2 L stores.
template <int NF>
__device__ __forceinline__ void dct_iv_pair(float* __restrict__ P, float2* __restrict__ X, const float2* __restrict__ dtw,
                                            const float2* __restrict__ ftw, int l, bool odd, bool live) {
    using namespace imdct_detail;
    using RP = RegFftPlan<NF / 2>;
    constexpr int N = NF / 2, R0 = RP::R0, R1 = RP::R1, G = RP::G, L = RP::L;
    static_assert(RP::half_warp, "both passes must fit half a warp");
    if (live && l < L) {
        float2 u[G];                                                  // stage 0 outputs, u[R0 * t1 + t0]
#pragma unroll
        for (int t1 = 0; t1 < R1; t1++) {
            float2 v[R0];
#pragma unroll
            for (int t0 = 0; t0 < R0; t0++) {
                // stage 0 butterfly l + L * t1, input t0: z[n] = dtw[n] * (x[2n] + i x[nf-1-2n]); the second half
                // loads the pair in the other order (even words for one frame, odd for the other: no bank conflicts)
                const int n = l + L * t1 + (N / R0) * t0;
                const float a = P[odd ? NF - 1 - 2 * n : 2 * n], b = P[odd ? 2 * n : NF - 1 - 2 * n];
                v[t0] = cmul(dtw[n], make_float2(odd ? b : a, odd ? a : b));
            }
            dft<R0>(v);
#pragma unroll
            for (int t0 = 0; t0 < R0; t0++) u[R0 * t1 + t0] = v[t0];
        }
#pragma unroll
        for (int k1 = 0; k1 < R0; k1++) {                             // stage 1 butterfly R0 * l + k1
            float2 v[R1];
#pragma unroll
            for (int t1 = 0; t1 < R1; t1++) {
                v[t1] = u[R0 * t1 + k1];
                if (t1 > 0) v[t1] = cmul(v[t1], ftw[k1 * t1 * L]);
            }
            dft<R1>(v);
#pragma unroll
            for (int t1 = 0; t1 < R1; t1++) X[G * l + k1 + R0 * t1] = v[t1];
        }
    }
    __syncwarp();
    if (live && l < G) {
        float2 x[L];
#pragma unroll
        for (int m = 0; m < L; m++) x[m] = X[G * m + l];
        column_stages<NF, 2, 1>(x, P, dtw, ftw, l, odd);
    }
    __syncwarp();
}

// Unfold (modified_dct.rs:97-136) and window: D holds the DCT-IV output; win[m] = gain * w[2nf-1-m].
// A lane's two consecutive samples (m, m + 1 with m even) are neighbours in D in all four segments of the unfolding
// (the segment borders nf/2, nf, 3nf/2 are even) and neighbours in the window, so each pair is one 8-byte shared-memory
// load and one 8-byte table load: the kernel is bound by the L1 / shared-memory path (MIO), not by arithmetic.
template <int NF, bool MS10>
__device__ __forceinline__ void imdct_unfold(const float* __restrict__ D, const float* __restrict__ win, int lane,
                                             float (&head)[2 * FrameGeo<NF, MS10>::NP], float (&tail)[2 * FrameGeo<NF, MS10>::NPT]) {
    using G = FrameGeo<NF, MS10>;
    constexpr int H = NF / 2, Z = G::Z;
    static_assert((H & 1) == 0 && (Z & 1) == 0 && (NF & 1) == 0, "pairs must not straddle a segment of the unfolding");
    auto t_pair = [&](int m) -> float2 {                                // (t[m], t[m + 1]) / gain, m even
        if (m < H) return *(const float2*)(D + H + m);
        if (m < NF) {
            const float2 q = *(const float2*)(D + (NF - 1 - (m - H)) - 1);
            return make_float2(-q.y, -q.x);
        }
        if (m < NF + H) {
            const float2 q = *(const float2*)(D + (H - 1 - (m - NF)) - 1);
            return make_float2(-q.y, -q.x);
        }
        const float2 q = *(const float2*)(D + (m - 3 * H));
        return make_float2(-q.x, -q.y);
    };
#pragma unroll
    for (int j = 0; j < G::NP; j++) {
        const int n = 64 * j + 2 * lane;
        if (64 * j + 64 <= NF || n < NF) {
            const float2 t = t_pair(Z + n), w = *(const float2*)(win + Z + n);
            head[2 * j] = __fmul_rn(t.x, w.x);
            head[2 * j + 1] = __fmul_rn(t.y, w.y);
        } else {
            head[2 * j] = 0.0f;
            head[2 * j + 1] = 0.0f;
        }
    }
#pragma unroll
    for (int j = 0; j < G::NPT; j++) {
        const int n = 64 * j + 2 * lane;
        if (64 * j + 64 <= NF - Z || n < NF - Z) {
            const float2 t = t_pair(NF + Z + n), w = *(const float2*)(win + NF + Z + n);
            tail[2 * j] = __fmul_rn(t.x, w.x);
            tail[2 * j + 1] = __fmul_rn(t.y, w.y);
        } else {
            tail[2 * j] = 0.0f;
            tail[2 * j + 1] = 0.0f;
        }
    }
}

// Call f.template operator()<NF, MS10>() for the frame geometry (nf, 10 ms?) of a configuration.
template <typename F>
inline bool dispatch_frame_geo(int nf, bool ms10, F&& f) {
    if (ms10) {
        switch (nf) {
            case 80: f.template operator()<80, true>(); return true;
            case 160: f.template operator()<160, true>(); return true;
            case 240: f.template operator()<240, true>(); return true;
            case 320: f.template operator()<320, true>(); return true;
            case 480: f.template operator()<480, true>(); return true;
        }
    } else {
        switch (nf) {
            case 60: f.template operator()<60, false>(); return true;
            case 120: f.template operator()<120, false>(); return true;
            case 180: f.template operator()<180, false>(); return true;
            case 240: f.template operator()<240, false>(); return true;
            case 360: f.template operator()<360, false>(); return true;
        }
    }
    return false;
}

}  // namespace lc3b
