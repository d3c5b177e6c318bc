// lc3b engine: time-parallel encode - many consecutive frames of every stream in ONE call (lc3b_encode_stream_frames).
//
// Of the encoder's per-stream state (EncoderState) only three groups really run along time:
//   * the attack envelope, the 50 Hz biquad of the LTPF analysis and its pitch / activation memory (enc_ltpf_kernel)
//   * the rate loop's offsets (ES_Q_*, enc_quantize_kernel)
// The MDCT time-buffer history of frame f is the tail of frame f - 1's own input, and everything else is a per-frame
// hand-off record between kernels.  So a call with F frames of S streams runs as S*F independent "units" through the
// unchanged kernels and touches the time axis only where it must:
//   1. enc_thist_prefill_kernel  each unit's MDCT history: the handle's for f = 0, else the previous frame's last nf - z samples
//   2. enc_mdct_kernel           over the S*F units (pcm row of unit s*F + f = frame f of stream s)
//   3. enc_thist_handback_kernel the last unit's history back into the handle
//   4. enc_ltpf_kernel           a warp per stream walks its F frames (per-stream state stays in the handle)
//   5. enc_sns_kernel, enc_tns_kernel over the units
//   6. enc_quantize_kernel       a warp per stream walks its F frames
//   7. bitstream prepare / range coder / finish over the units; unit s*F + f writes frames_out + (s*F + f)*frame_stride
// The per-frame buffers of the units live in the caller's scratch; the handle's own per-frame buffers (what
// lc3b_encoder_debug_read reports) are not touched.  Arithmetic is the frame-by-frame path's, so the bytes are identical.
#include "lc3b_enc_common.cuh"
#include "lc3b_plan.cuh"

namespace lc3b {

struct EncMultiLayout { size_t thist, xf, e_b, ehand, xq, qhand, lsbs, bs_scratch, total; };

static EncMultiLayout enc_multi_layout(const EncoderState& st, int F) {
    EncMultiLayout L;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = (off + bytes + 255) & ~(size_t)255; return o; };
    const lc3b_config& c = st.cfg;
    const size_t V = (size_t)st.n_streams * (size_t)F;
    L.thist = take(sizeof(int16_t) * V * (c.nf - c.z));
    L.xf = take(sizeof(float) * V * c.ne);
    L.e_b = take(sizeof(float) * V * 64);
    L.ehand = take(sizeof(int32_t) * V * EH_WORDS);
    L.xq = take(sizeof(int16_t) * V * c.ne);
    L.qhand = take(sizeof(int32_t) * V * QH_WORDS);
    L.lsbs = take(V * 2 * c.ne);
    L.bs_scratch = take(sizeof(uint32_t) * V * (size_t)st.bs_words);
    L.total = off;
    return L;
}

size_t enc_multi_scratch_bytes(const EncoderState& st, int n_frames) { return enc_multi_layout(st, n_frames).total; }

struct ThistParams {
    const int16_t* pcm;      // [S][F * nf]
    int16_t* hist;           // the handle's [S][nf - z]
    int16_t* thist_v;        // [S * F][nf - z]
    int S, F, nf, z;
};

// update_time_buffer (modified_dct.rs:126-138) keeps the last nf - z input samples: for unit (s, f > 0) those are
// pcm[s][(f - 1) nf + z, f nf), known before any kernel runs
__global__ void __launch_bounds__(256) enc_thist_prefill_kernel(ThistParams p) {
    const int L = p.nf - p.z;
    const size_t n_all = (size_t)p.S * p.F * L;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_all; i += (size_t)gridDim.x * blockDim.x) {
        const size_t v = i / L;
        const int n = (int)(i - v * L);
        const int f = (int)(v % p.F);
        p.thist_v[i] = f ? p.pcm[(v - 1) * p.nf + p.z + n] : p.hist[(v / p.F) * L + n];
    }
}

__global__ void __launch_bounds__(256) enc_thist_handback_kernel(ThistParams p) {
    const int L = p.nf - p.z;
    const size_t n_all = (size_t)p.S * L;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_all; i += (size_t)gridDim.x * blockDim.x) {
        const size_t s = i / L;
        p.hist[i] = p.thist_v[((s + 1) * p.F - 1) * L + (i - s * L)];
    }
}

static unsigned copy_grid(size_t n) {
    const size_t g = (n + 255) / 256;
    return (unsigned)(g < 4096 ? g : 4096);
}

void plan_enc_multi(LaunchPlan& plan, const EncoderState& st, const int16_t* pcm, int n_frames, uint8_t* frames_out, int nbytes,
                    size_t frame_stride, void* scratch) {
    const int S = st.n_streams, F = n_frames;
    const EncMultiLayout L = enc_multi_layout(st, F);
    uint8_t* base = (uint8_t*)scratch;
    // a view of the handle with S*F units: per-frame buffers in the scratch, per-stream state the handle's
    EncoderState vs = st;
    vs.n_streams = S * F;
    vs.thist = (int16_t*)(base + L.thist);
    vs.xf = (float*)(base + L.xf);
    vs.e_b = (float*)(base + L.e_b);
    vs.ehand = (int32_t*)(base + L.ehand);
    vs.xq = (int16_t*)(base + L.xq);
    vs.qhand = (int32_t*)(base + L.qhand);
    vs.lsbs = base + L.lsbs;
    vs.bs_scratch = (uint32_t*)(base + L.bs_scratch);
    const ThistParams tp{pcm, st.thist, vs.thist, S, F, st.cfg.nf, st.cfg.z};
    const size_t hist_len = (size_t)(st.cfg.nf - st.cfg.z);
    const size_t nf = (size_t)st.cfg.nf;
    plan.add(enc_thist_prefill_kernel, copy_grid((size_t)S * F * hist_len), 256, 0, tp);
    plan_enc_analysis(plan, vs, pcm, nf, nbytes, 1, F);
    plan.add(enc_thist_handback_kernel, copy_grid((size_t)S * hist_len), 256, 0, tp);
    plan_enc_analysis(plan, vs, pcm, nf, nbytes, 2, F);
    plan_enc_quant(plan, vs, frames_out, nbytes, frame_stride, 15, F);
}

}  // namespace lc3b
