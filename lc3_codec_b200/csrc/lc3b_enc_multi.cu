// lc3b engine: time-parallel encode - many consecutive frames of many streams in ONE call (lc3b_encode_stream_frames and
// lc3b_encode_stream_frames_subset).
//
// Of the encoder's per-stream state (EncoderState) only three groups really run along time:
//   * the attack envelope, the 50 Hz biquad of the LTPF analysis and its pitch / activation memory (enc_ltpf_kernel)
//   * the rate loop's offsets (ES_Q_*, enc_quantize_kernel)
// The MDCT time-buffer history of frame f is the tail of frame f - 1's own input, and everything else is a per-frame
// hand-off record between kernels.  A call lists rows in a row table (lc3b_common.cuh): row i advances handle stream row_i
// by count_i consecutive frames, units off_i .. off_i + count_i - 1.  The subset call sends its table; the dense call is
// the identity table of S rows of F frames, which unit_rows_kernel writes on the device.  The units run independently
// through the unchanged kernels and the time axis is touched only where it must be:
//   0. unit_rows_kernel          unit_row[v], the state row of each unit's row (plan_unit_rows, lc3b_dec_multi.cu)
//   1. enc_thist_prefill_kernel  each unit's MDCT history: the handle's for a row's first unit, else the previous frame's
//                                last nf - z samples
//   2. enc_mdct_kernel           over the units (pcm row v = unit v)
//   3. enc_thist_handback_kernel each row's last unit's history back into the handle
//   4. enc_ltpf_kernel           a warp per row walks its frames (per-stream state stays in the handle)
//   5. enc_sns_kernel, enc_tns_kernel over the units
//   6. enc_quantize_kernel       a warp per row walks its frames
//   7. bitstream prepare / range coder / finish over the units; unit v writes frames_out + v * frame_stride
// The per-frame buffers of the units live in the caller's scratch; the handle's own per-frame buffers (what
// lc3b_encoder_debug_read reports) are not touched.  Arithmetic is the frame-by-frame path's, so the bytes are identical.
#include "lc3b_enc_common.cuh"
#include "lc3b_plan.cuh"

namespace lc3b {

struct EncMultiLayout { size_t rows, thist, xf, e_b, ehand, xq, qhand, lsbs, bs_scratch, unit_row, total; };

// V units of n_rows rows: the row table at the front (where RowTable::send puts it) and unit_row[V] at the end
static EncMultiLayout enc_multi_layout(const EncoderState& st, int n_rows, size_t V) {
    EncMultiLayout L;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = (off + bytes + 255) & ~(size_t)255; return o; };
    const lc3b_config& c = st.cfg;
    L.rows = take(sizeof(int32_t) * RT_WORDS * n_rows);
    L.thist = take(sizeof(int16_t) * V * (c.nf - c.z));
    L.xf = take(sizeof(float) * V * c.ne);
    L.e_b = take(sizeof(float) * V * 64);
    L.ehand = take(sizeof(int32_t) * V * EH_WORDS);
    L.xq = take(sizeof(int16_t) * V * c.ne);
    L.qhand = take(sizeof(int32_t) * V * QH_WORDS);
    L.lsbs = take(V * 2 * c.ne);
    L.bs_scratch = take(sizeof(uint32_t) * V * (size_t)st.bs_words);
    L.unit_row = take(sizeof(int32_t) * V);
    L.total = off;
    return L;
}

size_t enc_multi_scratch_bytes(const EncoderState& st, int n_rows, long long total) {
    return enc_multi_layout(st, n_rows, (size_t)total).total;
}

struct ThistParams {
    const int16_t* pcm;      // [V][nf]
    int16_t* hist;           // the handle's [S][nf - z]
    int16_t* thist_v;        // [V][nf - z]
    int n_rows, nf, z;       // rows of the row table
    const int32_t* rows;
    const int32_t* unit_row; // [V] the state row of unit v's row, ~row for its first unit
    size_t V;
};

// update_time_buffer (modified_dct.rs:126-138) keeps the last nf - z input samples: for a unit v that is not its row's
// first, those are pcm[(v - 1) nf + z, v nf), known before any kernel runs
__global__ void __launch_bounds__(256) enc_thist_prefill_kernel(ThistParams p) {
    const int L = p.nf - p.z;
    const size_t n_all = p.V * L;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_all; i += (size_t)gridDim.x * blockDim.x) {
        const size_t v = i / L;
        const int n = (int)(i - v * L);
        const int u = p.unit_row[v];
        p.thist_v[i] = u >= 0 ? p.pcm[(v - 1) * p.nf + p.z + n] : p.hist[(size_t)~u * L + n];
    }
}

// the history of each row's last unit back to its state row
__global__ void __launch_bounds__(256) enc_thist_handback_kernel(ThistParams p) {
    const int L = p.nf - p.z;
    const size_t n_all = (size_t)p.n_rows * L;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_all; i += (size_t)gridDim.x * blockDim.x) {
        const size_t s = i / L;
        const RowSpan rs = row_span(p.rows, (int)s);
        p.hist[(size_t)rs.row * L + (i - s * L)] = p.thist_v[((size_t)rs.off + rs.count - 1) * L + (i - s * L)];
    }
}

static unsigned copy_grid(size_t n) {
    const size_t g = (n + 255) / 256;
    return (unsigned)(g < 4096 ? g : 4096);
}

void plan_enc_multi(LaunchPlan& plan, const EncoderState& st, const int16_t* pcm, int n_rows, int n_live, long long total,
                    int dense_frames, uint8_t* frames_out, int nbytes, size_t frame_stride, void* scratch) {
    const size_t V = (size_t)total;
    const EncMultiLayout L = enc_multi_layout(st, n_rows, V);
    uint8_t* base = (uint8_t*)scratch;
    // a view of the handle with V units: per-frame buffers in the scratch, per-stream state the handle's
    EncoderState vs = st;
    vs.n_streams = (int)V;
    vs.thist = (int16_t*)(base + L.thist);
    vs.xf = (float*)(base + L.xf);
    vs.e_b = (float*)(base + L.e_b);
    vs.ehand = (int32_t*)(base + L.ehand);
    vs.xq = (int16_t*)(base + L.xq);
    vs.qhand = (int32_t*)(base + L.qhand);
    vs.lsbs = base + L.lsbs;
    vs.bs_scratch = (uint32_t*)(base + L.bs_scratch);
    const size_t hist_len = (size_t)(st.cfg.nf - st.cfg.z);
    const size_t nf = (size_t)st.cfg.nf;
    int32_t* rows = (int32_t*)(base + L.rows);
    int32_t* unit_row = (int32_t*)(base + L.unit_row);
    const ThistParams tp{pcm, st.thist, vs.thist, n_live, st.cfg.nf, st.cfg.z, rows, unit_row, V};
    plan_unit_rows(plan, rows, n_live, dense_frames, unit_row);
    plan.add(enc_thist_prefill_kernel, copy_grid(V * hist_len), 256, 0, tp);
    plan_enc_analysis(plan, vs, pcm, nf, nbytes, 1);
    plan.add(enc_thist_handback_kernel, copy_grid((size_t)n_live * hist_len), 256, 0, tp);
    plan_enc_analysis(plan, vs, pcm, nf, nbytes, 2, nullptr, rows, n_live);
    plan_enc_quant(plan, vs, frames_out, nbytes, frame_stride, 15, nullptr, rows, n_live);
}

}  // namespace lc3b
