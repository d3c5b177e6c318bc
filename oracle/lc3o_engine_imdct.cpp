// CPU ORACLE - TEST INFRASTRUCTURE (see lc3o.h).
// The CUDA engine's inverse MDCT, restated op for op so that the oracle can run the decoder with the engine's transform
// (DecMdct with EngineImdct) and the engine's PCM can be compared with it bit for bit:
//
//   dct_iv_warp / stage<> / dft<R> / cmul   lc3_codec_b200/csrc/lc3b_imdct.cuh (FftPlan, Stockham index maps)
//   imdct_unfold                            lc3_codec_b200/csrc/lc3b_imdct.cuh (t_pair segments, folded window)
//   win / dtw / ftw tables                  lc3_codec_b200/csrc/lc3b_api.cu init_tables_kernel
//
// The kernel's __fmaf_rn is std::fmaf here and its __fmul_rn / __fadd_rn / __fsub_rn are plain * + -, which the oracle's
// -ffp-contract=off keeps unfused.  The engine's FFT factors N = nf / 2 differently from kissfft (radix 5 first, then 3s,
// 4s, 2), so this transform and DctIv differ in their last bits; tests/test_engine_transform_cpu.py bounds both against a
// float64 DCT-IV.  Everything around the transform (concealment, overlap-add, post filter, rounding) stays the oracle's.
#include "lc3o.h"

namespace lc3o {

namespace {

Cpx e_cmul(Cpx a, Cpx b) { return {std::fmaf(a.r, b.r, -(a.i * b.i)), std::fmaf(a.r, b.i, a.i * b.r)}; }
Cpx e_cadd(Cpx a, Cpx b) { return {a.r + b.r, a.i + b.i}; }
Cpx e_csub(Cpx a, Cpx b) { return {a.r - b.r, a.i - b.i}; }

void e_dft2(Cpx* v) {
    const Cpx a = v[0], b = v[1];
    v[0] = e_cadd(a, b);
    v[1] = e_csub(a, b);
}
void e_dft3(Cpx* v) {
    const float S = 0.86602540378443864676f;
    const Cpx t = e_cadd(v[1], v[2]), d = e_csub(v[1], v[2]);
    const Cpx m = {std::fmaf(-0.5f, t.r, v[0].r), std::fmaf(-0.5f, t.i, v[0].i)};
    const Cpx r = {S * d.i, -(S * d.r)};
    v[0] = e_cadd(v[0], t);
    v[1] = e_cadd(m, r);
    v[2] = e_csub(m, r);
}
void e_dft4(Cpx* v) {
    const Cpx a = e_cadd(v[0], v[2]), b = e_csub(v[0], v[2]);
    const Cpx c = e_cadd(v[1], v[3]), d = e_csub(v[1], v[3]);
    const Cpx dj = {d.i, -d.r};
    v[0] = e_cadd(a, c);
    v[1] = e_cadd(b, dj);
    v[2] = e_csub(a, c);
    v[3] = e_csub(b, dj);
}
void e_dft5(Cpx* v) {
    const float C1 = 0.30901699437494742410f, C2 = -0.80901699437494742410f;
    const float S1 = 0.95105651629515357212f, S2 = 0.58778525229247312917f;
    const Cpx a1 = e_cadd(v[1], v[4]), b1 = e_csub(v[1], v[4]);
    const Cpx a2 = e_cadd(v[2], v[3]), b2 = e_csub(v[2], v[3]);
    const Cpx m1 = {std::fmaf(C2, a2.r, std::fmaf(C1, a1.r, v[0].r)), std::fmaf(C2, a2.i, std::fmaf(C1, a1.i, v[0].i))};
    const Cpx m2 = {std::fmaf(C1, a2.r, std::fmaf(C2, a1.r, v[0].r)), std::fmaf(C1, a2.i, std::fmaf(C2, a1.i, v[0].i))};
    const Cpx n1 = {std::fmaf(S2, b2.i, S1 * b1.i), -std::fmaf(S2, b2.r, S1 * b1.r)};
    const Cpx n2 = {std::fmaf(-S1, b2.i, S2 * b1.i), -std::fmaf(-S1, b2.r, S2 * b1.r)};
    v[0] = {(v[0].r + a1.r) + a2.r, (v[0].i + a1.i) + a2.i};
    v[1] = e_cadd(m1, n1);
    v[4] = e_csub(m1, n1);
    v[2] = e_cadd(m2, n2);
    v[3] = e_csub(m2, n2);
}
void e_dft(int R, Cpx* v) {
    switch (R) {
        case 2: e_dft2(v); break;
        case 3: e_dft3(v); break;
        case 4: e_dft4(v); break;
        default: e_dft5(v); break;
    }
}

}  // namespace

// lc3b_imdct.cuh FftPlan<N>
bool EngineImdct::plan(int n, int* radices, int* count) {
    static const struct { int n, k, r[4]; } P[] = {
        {30, 3, {5, 3, 2, 0}},  {40, 3, {5, 4, 2, 0}},  {60, 3, {5, 3, 4, 0}},  {80, 3, {5, 4, 4, 0}},  {90, 4, {5, 3, 3, 2}},
        {120, 4, {5, 3, 4, 2}}, {160, 4, {5, 4, 4, 2}}, {180, 4, {5, 3, 3, 4}}, {240, 4, {5, 3, 4, 4}}};
    for (const auto& p : P) {
        if (p.n != n) continue;
        *count = p.k;
        for (int i = 0; i < p.k; i++) radices[i] = p.r[i];
        return true;
    }
    return false;
}

// lc3b_api.cu init_tables_kernel: f64 angles narrowed to f32, the window folded with the 1 / sqrt(2 nf) gain
void EngineImdct::init(const Config& c) {
    nf = c.nf;
    z = c.z;
    const int N = nf / 2;
    plan(N, radices, &n_stages);
    dtw.resize(N);
    ftw.resize(N);
    for (int i = 0; i < N; i++) {
        const double t = -M_PI * (double)(8 * i + 1) / (8.0 * (double)N * 2.0);
        dtw[i] = {(float)std::cos(t), (float)std::sin(t)};
        const double ph = -2.0 * M_PI * (double)i / (double)N;
        ftw[i] = {(float)std::cos(ph), (float)std::sin(ph)};
    }
    const float* w = mdct_window(c);
    const float gain = 1.0f / std::sqrt(2.0f * (float)nf);
    win.resize(2 * nf);
    for (int m = 0; m < 2 * nf; m++) win[m] = gain * w[2 * nf - 1 - m];
    p.assign(nf, 0.0f);
    q.assign(nf, 0.0f);
}

// lc3b_imdct.cuh dct_iv_warp: stage s reads one buffer and writes the other; the first stage applies the DCT-IV
// pre-twiddle to the real input, the last the post-twiddle, scattering nf real coefficients
void EngineImdct::dct_iv(float* buf) {
    const int N = nf / 2;
    std::memcpy(p.data(), buf, sizeof(float) * nf);
    float* src = p.data();
    float* dst = q.data();
    int NS = 1;
    for (int s = 0; s < n_stages; s++) {
        const int R = radices[s], NBF = N / R, TW = N / (NS * R);
        const bool first = s == 0, last = s == n_stages - 1;
        for (int j = 0; j < NBF; j++) {
            const int k = j % NS;
            Cpx v[5];
            for (int t = 0; t < R; t++) {
                const int n = j + t * NBF;
                if (first) v[t] = e_cmul(dtw[n], Cpx{src[2 * n], src[nf - 1 - 2 * n]});
                else {
                    v[t] = Cpx{src[2 * n], src[2 * n + 1]};
                    if (t > 0 && NS > 1) v[t] = e_cmul(v[t], ftw[k * t * TW]);
                }
            }
            e_dft(R, v);
            const int base = (j - k) * R + k;
            for (int t = 0; t < R; t++) {
                const int o = base + t * NS;
                if (last) {
                    const Cpx w = e_cmul(dtw[o], v[t]);
                    dst[2 * o] = w.r * 2.0f;
                    dst[nf - 1 - 2 * o] = w.i * -2.0f;
                } else {
                    dst[2 * o] = v[t].r;
                    dst[2 * o + 1] = v[t].i;
                }
            }
        }
        NS *= R;
        std::swap(src, dst);
    }
    std::memcpy(buf, src, sizeof(float) * nf);
}

// lc3b_imdct.cuh imdct_unfold: head[n] = t[z + n] * win[z + n] (n < nf), tail[n] = t[nf + z + n] * win[nf + z + n]
// (n < nf - z), where t / gain is the DCT-IV output D unfolded (modified_dct.rs:97-136) segment by segment
void EngineImdct::unfold(const float* D, float* head, float* tail) const {
    const int H = nf / 2;
    auto t_of = [&](int m) -> float {
        if (m < H) return D[H + m];
        if (m < nf) return -D[nf - 1 - (m - H)];
        if (m < nf + H) return -D[H - 1 - (m - nf)];
        return -D[m - 3 * H];
    };
    for (int n = 0; n < nf; n++) head[n] = t_of(z + n) * win[z + n];
    for (int n = 0; n < nf - z; n++) tail[n] = t_of(nf + z + n) * win[nf + z + n];
}

}  // namespace lc3o
