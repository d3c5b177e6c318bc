// lc3b engine, decoder kernels 2 and 3: shaped spectrum -> PCM, one WARP per frame (two at nf = 480, large batches).
//
// Replaces, per stream, the second half of DecoderChannel::decode (src/decoder/lc3_decoder.rs:134-153):
//   PacketLossConcealment::save / load_into   src/decoder/packet_loss_concealment.rs:50,63
//   ModDiscreteCosTrans::run                  src/decoder/modified_dct.rs:76 (DCT-IV via N = nf/2 complex FFT,
//                                             src/common/dct_iv.rs:49, src/common/kissfft.rs:78; window; overlap-add)
//   LongTermPostFilter::run                   src/decoder/long_term_post_filter.rs:252 (five transition cases)
//   output_scaling::scale_and_round           src/decoder/output_scaling.rs:13
// Concealment, post filter and rounding are shared with the time-parallel path (lc3b_synth.cuh), the inverse MDCT too
// (lc3b_imdct.cuh).
//
// synth_classic_kernel<NF, MS10> (every stream, the default): concealment, inverse MDCT (frame length a template
// constant), overlap-add, and the post filter's PASS-THROUGH case: x_hat goes to the LTPF history ring and, rounded, to
// the PCM row.  Two consecutive samples per lane, so PCM leaves as 32-bit and f32 state as 64-bit accesses; all global
// traffic is stream-major and coalesced (spectrum 4*ne B in, overlap memory 4*(nf-z) B in/out, LTPF history 4*nf B
// out, PCM 2*nf B out).  synth_pair_kernel<480, true> is the same work with two frames per warp and the FFT in registers
// (large batches at 48 / 44.1 kHz, 10 ms); synth mode 1 (lc3b_decoder_set_synth_mode) keeps synth_classic_kernel there
// too.  Both give the same bits.
// ltpf_kernel (streams whose post filter is, or was in the previous frame, active): the IIR itself; for those streams
// the synthesis kernel leaves x_hat in a side buffer (the ring block keeps the samples long pitch lags still reach), and
// this kernel writes the filtered signal to the ring block and the PCM row.  Streams outside such a span cost this
// kernel one flag load.
#include <string.h>

#include "lc3b_common.cuh"
#include "lc3b_imdct.cuh"
#include "lc3b_math.cuh"
#include "lc3b_plan.cuh"
#include "lc3b_synth.cuh"

namespace lc3b {

struct SynthParams {
    const DevConfig* cfg;
    const float* win;
    const float2* dtw;
    const float2* ftw;
    const float* spec;
    float* ola;
    float* ltpf_y;
    float* ltpf_xtail;
    float* ltpf_x;       // [n_streams][nf] x_hat of streams inside an active span (synthesis kernel -> ltpf_kernel)
    int32_t* side;
    int32_t* sstate;
    int16_t* pcm_out;
    size_t pcm_stride;
    int n_streams;       // streams of this launch (a sub-batch when a call is split)
    int slot_streams;    // streams per spectrum slot = the handle's stream count
    int hist_len;        // ltpf_blocks * nf
    int pcm_pairs;       // PCM rows are 4-byte aligned: samples leave two at a time
    int group;           // ltpf_kernel: streams looked after by one warp
    int smem_per_warp;   // ltpf_kernel, bytes
    int no_ltpf;         // the handle's minimum frame length rules the post filter out: no history is kept (lc3b_decoder_set_min_nbytes)
    const int32_t* ids;  // subset call: row u of this launch is handle stream ids[u] (the IDS instantiations only)
};

constexpr int SYN_WARPS = 4;

// synth_classic_kernel: one warp = one frame, spectrum through ordinary loads.  What bounds it is the SM's L1 /
// shared-memory data path, not instruction issue, DRAM or latency: dropping a quarter of its instructions (the float ->
// int casts) changed nothing, the time per frame is the same at 16 384 streams (everything in L2) as at 262 144, MORE
// resident warps make it slower (8 / 10 / 12 CTAs per SM: 0.502 / 0.516 / 0.529 ms - the twiddle and window tables share
// L1 with the shared-memory carve-out), and a persistent variant that prefetched the next frame's spectrum with the TMA
// unit was slower still (0.525 against 0.50 ms at 262 144 streams, profiles/r2_synth_ab.json, DESIGN.md §3).  The
// per-frame streams (spectrum, overlap memory, PCM) therefore use evict-first loads and stores, which leaves L1 to the
// tables (0.517 -> 0.500 ms).
//
// synth_pair_kernel: the same work with two frames per warp (rows 2w and 2w + 1), at 48 / 44.1 kHz, 10 ms (nf = 480)
// only.  The two frames are transformed together by dct_iv_pair, one per half warp: the FFT stays in registers but for
// one exchange through shared memory, and every table load and shared-memory instruction of the transform serves both
// frames (per frame: 45 -> 23 shared loads, 43 -> 23.5 shared stores, 36 -> 26.5 table loads).  Everything else
// (spectrum load, concealment, unfold, overlap-add, history, PCM) runs one frame at a time on the whole warp.  A pair
// warp is a longer serial chain than a single-frame warp, so small launches, which are latency bound, keep
// synth_classic_kernel (the row threshold is in PlanSynth::add).
template <int NF>
constexpr bool synth_pairs() { return NF == 480; }
constexpr int SYN_PAIR_CTAS = 5;      // CTAs per SM the pair kernel is compiled for (96 registers; 4 CTAs at 104: 0.400 ms, 5: 0.358)

// One warp's FPW frames: the body of both kernels.
template <int NF, bool MS10, bool IDS, int FPW>
__device__ __forceinline__ void synth_frames(const SynthParams& p) {
    using G = FrameGeo<NF, MS10>;
    constexpr int NE = G::NE, Z = G::Z, NP = G::NP, NPT = G::NPT;
    extern __shared__ __align__(16) uint8_t smem[];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int row0 = (blockIdx.x * SYN_WARPS + wid) * FPW;
    if (row0 >= p.n_streams) return;                              // warps are independent: no CTA-wide barrier below

    // per frame f of the warp: P = spectrum in, FFT ping (and the output of dct_iv_pair); Q = FFT pong / exchange
    float* const W = (float*)smem + (size_t)wid * FPW * 2 * NF;
    auto P = [&](int f) { return W + f * NF; };
    auto Q = [&](int f) { return W + (FPW + f) * NF; };

    // what a frame needs after the transform
    int stream[FPW], active[FPW], prev_active[FPW], blk_idx[FPW];
    int32_t *sd[FPW], *ss[FPW];
    float* ola[FPW];
    float2 ola_r[FPW][NPT];
#pragma unroll
    for (int f = 0; f < FPW; f++) {
        if (f > 0 && row0 + f >= p.n_streams) break;              // an odd row count: the last warp has one frame
        const int s = stream[f] = state_row<IDS>(p.ids, row0 + f);   // persistent rows; PCM goes to the call's row
        sd[f] = p.side + (size_t)s * SIDE_WORDS;
        ss[f] = p.sstate + (size_t)s * SS_WORDS;
        // the two records as 16-byte loads (every lane reads the same words; each load is one slot of the memory pipe)
        static_assert(SD_OK == 0 && SD_LTPF_ACTIVE == 1 && SD_SLOT == 6 && SS_PLC_LOST == 1 && SS_PLC_ALPHA == 2 && SS_LTPF_PREV == 4 &&
                          SS_LTPF_BLK == 7,
                      "record layout");
        const int4 sd_a = ((const int4*)sd[f])[0], sd_b = ((const int4*)sd[f])[1];
        const int4 ss_a = ((const int4*)ss[f])[0], ss_b = ((const int4*)ss[f])[1];
        const int ok = sd_a.x;
        const int slot = sd_b.z;
        active[f] = sd_a.y;
        prev_active[f] = ltpf_prev_active(ss_b.x);
        blk_idx[f] = ss_b.w;
        const float* sp = p.spec + ((size_t)slot * p.slot_streams + s) * NE;

        // overlap memory: requested now, consumed after the FFT
        ola[f] = p.ola + (size_t)s * (NF - Z);
#pragma unroll
        for (int j = 0; j < NPT; j++)
            ola_r[f][j] = (64 * j + 64 <= NF - Z || 64 * j + 2 * lane < NF - Z) ? __ldcs((const float2*)ola[f] + 32 * j + lane) : make_float2(0.0f, 0.0f);

        // ---- spectrum load, with concealment (packet_loss_concealment.rs:63-85) when the frame was bad
        if (ok) {
#pragma unroll
            for (int k0 = 0; k0 < NF / 4; k0 += 32) {
                const int k4 = k0 + lane;
                if (k0 + 32 <= NF / 4 || k4 < NF / 4)
                    ((float4*)P(f))[k4] = 4 * k4 < NE ? __ldcs((const float4*)sp + k4) : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
            }
            if (lane == 0 && (ss_a.y != 0 || ss_a.z != (int32_t)f2u(1.0f))) { ss[f][SS_PLC_LOST] = 0; ss[f][SS_PLC_ALPHA] = (int32_t)f2u(1.0f); }
        } else {
            const int lost = ss_a.y;
            float alpha = u2f((uint32_t)ss_a.z);
            __syncwarp();                                        // every lane has read the state before any lane updates it
            alpha = plc_fade(alpha, lost);
            plc_scramble<NF, NE>(P(f), sp, alpha, (uint32_t)ss_a.w, lane, ss[f] + SS_PLC_SEED);
            if (lane == 0) { ss[f][SS_PLC_LOST] = lost + 1; ss[f][SS_PLC_ALPHA] = (int32_t)f2u(alpha); }
        }
    }
    __syncwarp();

    // ---- DCT-IV (dct_iv.rs:49-67)
    const float* D0;                                              // where frame 0's coefficients are (frame 1's: in P(1))
    if constexpr (FPW == 2) {
        const int h = lane >> 4;
        dct_iv_pair<NF>(P(h), (float2*)Q(h), p.dtw, p.ftw, lane & 15, h == 1, row0 + h < p.n_streams);
        D0 = P(0);
    } else D0 = dct_iv_warp<NF>(P(0), Q(0), p.dtw, p.ftw, lane);

#pragma unroll
    for (int f = 0; f < FPW; f++) {
        if (f > 0 && row0 + f >= p.n_streams) break;
        const int s = stream[f];
        // with two frames the per-stream pointers are derived again rather than held through the transform (registers)
        float* const ola_f = FPW == 1 ? ola[f] : p.ola + (size_t)s * (NF - Z);
        int32_t* const sd_f = FPW == 1 ? sd[f] : p.side + (size_t)s * SIDE_WORDS;
        int32_t* const ss_f = FPW == 1 ? ss[f] : p.sstate + (size_t)s * SS_WORDS;
        // ---- unfold, window (modified_dct.rs:97-136)
        float head[2 * NP], tail[2 * NPT];
        imdct_unfold<NF, MS10>(f == 0 ? D0 : P(f), p.win, lane, head, tail);

        // ---- overlap-add (modified_dct.rs:138-151): two roundings, like the reference (and the time-parallel path)
#pragma unroll
        for (int j = 0; j < NPT; j++) {
            if (64 * j + 64 <= NF - Z || 64 * j + 2 * lane < NF - Z) {
                head[2 * j] = xa(ola_r[f][j].x, head[2 * j]);
                head[2 * j + 1] = xa(ola_r[f][j].y, head[2 * j + 1]);
                __stcs((float2*)ola_f + 32 * j + lane, make_float2(tail[2 * j], tail[2 * j + 1]));
            }
        }

        // ---- post filter, pass-through case (long_term_post_filter.rs:252-343 with zero coefficients): history + PCM
        // Inside an active span the ring block must keep its old content until the filter has run (long pitch lags reach
        // around the ring into it), so x_hat waits in a side buffer for ltpf_kernel instead.
        const bool in_span = active[f] || prev_active[f];
        const int blk = blk_idx[f];
        float* yblk = in_span ? p.ltpf_x + (size_t)s * NF : p.ltpf_y + (size_t)s * p.hist_len + blk * NF;
        float* xtail = p.ltpf_xtail + (size_t)s * XTAIL_FLOATS + blk * 16;
        int16_t* out = p.pcm_out + (size_t)(row0 + f) * p.pcm_stride;
#pragma unroll
        for (int j = 0; j < NP; j++) {
            const int n = 64 * j + 2 * lane;
            if (64 * j + 64 <= NF || n < NF) {
                const float a = head[2 * j], b = head[2 * j + 1];
                if (!p.no_ltpf) {
                    ((float2*)yblk)[32 * j + lane] = make_float2(a, b);
                    if (n >= NF - 16) ((float2*)xtail)[(n - (NF - 16)) >> 1] = make_float2(a, b);   // x_hat tail for the next frame's filter
                }
                const int32_t qa = round_pcm_i32(a), qb = round_pcm_i32(b);
                if (p.pcm_pairs) __stcs((uint32_t*)out + 32 * j + lane, ((uint32_t)qa & 0xffffu) | ((uint32_t)qb << 16));
                else { out[n] = (int16_t)qa; out[n + 1] = (int16_t)qb; }
            }
        }
        if (lane == 0 && !p.no_ltpf) {
            sd_f[SD_BLK] = blk;
            int nb = blk + 1;                                    // :334-337
            if (nb > (MS10 ? 1 : 2)) nb = 0;
            ss_f[SS_LTPF_BLK] = nb;
            if (!in_span) ltpf_store_prev(ss_f, LtpfPar{});     // otherwise ltpf_kernel carries the filter state on
        }
    }
}

template <int NF, bool MS10, bool IDS>
__global__ void __launch_bounds__(SYN_WARPS * 32) synth_classic_kernel(const __grid_constant__ SynthParams p) {
    synth_frames<NF, MS10, IDS, 1>(p);
}
template <int NF, bool MS10, bool IDS>
__global__ void __launch_bounds__(SYN_WARPS * 32, SYN_PAIR_CTAS) synth_pair_kernel(const __grid_constant__ SynthParams p) {
    synth_frames<NF, MS10, IDS, 2>(p);
}
// shared memory of both kernels: per warp two nf-float buffers per frame
constexpr int synth_warp_smem_bytes(int nf, int fpw) { return SYN_WARPS * fpw * 2 * nf * 4; }

// ---------------------------------------------------------------- kernel 3: the post filter where it is not idle
template <bool IDS>
__global__ void __launch_bounds__(SYN_WARPS * 32) ltpf_kernel(SynthParams p) {
    extern __shared__ __align__(16) uint8_t smem[];
    const DevConfig& c = *p.cfg;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int first = (blockIdx.x * SYN_WARPS + wid) * p.group;
    if (first >= p.n_streams) return;
    // which streams of this warp's group are inside an active span
    uint32_t todo;
    {
        const int r = first + lane;
        bool in_span = false;
        if (lane < p.group && r < p.n_streams) {
            const int s = state_row<IDS>(p.ids, r);
            in_span = p.side[(size_t)s * SIDE_WORDS + SD_LTPF_ACTIVE] != 0 || ltpf_prev_active(p.sstate[(size_t)s * SS_WORDS + SS_LTPF_PREV]);
        }
        todo = __ballot_sync(0xffffffffu, in_span);
    }
    if (todo == 0) return;
    const LtpfGeo g = ltpf_geo(c, p.hist_len);
    const int nf = g.nf, blocks = g.blocks;
    float* Y = (float*)(smem + (size_t)wid * p.smem_per_warp);    // per-warp buffer, see ltpf_warp_bytes
    float* X = Y + p.hist_len;
    float* xt = X + nf;
    float* scratch = xt + 16;

    while (todo) {
        const int row = first + (__ffs(todo) - 1);
        const int stream = state_row<IDS>(p.ids, row);
        todo &= todo - 1;
        const int32_t* sd = p.side + (size_t)stream * SIDE_WORDS;
        int32_t* ss = p.sstate + (size_t)stream * SS_WORDS;
        const LtpfPar cur = ltpf_params(c, sd), prev = ltpf_load_prev(ss);
        const int blk_idx = sd[SD_BLK];
        const int blk = blk_idx * nf;
        float* yhist = p.ltpf_y + (size_t)stream * p.hist_len;
        const float* xtail_prev = p.ltpf_xtail + (size_t)stream * XTAIL_FLOATS + (blk_idx == 0 ? blocks - 1 : blk_idx - 1) * 16;
        __syncwarp();                                  // the previous stream's reads of the shared buffers are done
        for (int n = lane; n < p.hist_len; n += 32) Y[n] = yhist[n];
        if (lane < 16) xt[lane] = xtail_prev[lane];
        __syncwarp();
        for (int n = lane; n < nf; n += 32) X[n] = p.ltpf_x[(size_t)stream * nf + n];   // x_hat left by the synthesis kernel
        __syncwarp();
        ltpf_filter_frame(c, g, Y, X, xt, scratch, blk, cur, prev, lane);
        int16_t* out = p.pcm_out + (size_t)row * p.pcm_stride;
        for (int n = lane; n < nf; n += 32) {
            const float v = Y[blk + n];
            yhist[blk + n] = v;
            out[n] = (int16_t)round_pcm_i32(v);
        }
        if (lane == 0) ltpf_store_prev(ss, cur);
    }
}

namespace {
struct PrepareSynth {
    cudaError_t e = cudaSuccess;
    template <int NF, bool MS10> void operator()() {
        e = cudaFuncSetAttribute(synth_classic_kernel<NF, MS10, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, synth_warp_smem_bytes(NF, 1));
        if (e == cudaSuccess) e = cudaFuncSetAttribute(synth_classic_kernel<NF, MS10, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, synth_warp_smem_bytes(NF, 1));
        if constexpr (synth_pairs<NF>()) {
            if (e == cudaSuccess) e = cudaFuncSetAttribute(synth_pair_kernel<NF, MS10, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, synth_warp_smem_bytes(NF, 2));
            if (e == cudaSuccess) e = cudaFuncSetAttribute(synth_pair_kernel<NF, MS10, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, synth_warp_smem_bytes(NF, 2));
        }
    }
};
struct PlanSynth {
    LaunchPlan& plan;
    const SynthParams& p;
    int dep, node, sm_count;
    bool single;         // synth mode 1: one frame per warp at every size
    template <int NF, bool MS10> void operator()() {
        if (p.ids) add<NF, MS10, true>();
        else add<NF, MS10, false>();
    }
    template <int NF, bool MS10, bool IDS> void add() {
        if constexpr (synth_pairs<NF>()) {
            // two frames per warp once the launch fills every SM with pair warps twice over; below that the launch is
            // latency bound and one frame per warp, twice the warps, finishes sooner
            if (!single && p.n_streams >= 2 * sm_count * SYN_PAIR_CTAS * SYN_WARPS * 2) {
                node = plan.add(synth_pair_kernel<NF, MS10, IDS>, (unsigned)((p.n_streams + 2 * SYN_WARPS - 1) / (2 * SYN_WARPS)), SYN_WARPS * 32,
                                synth_warp_smem_bytes(NF, 2), p, dep);
                return;
            }
        }
        node = plan.add(synth_classic_kernel<NF, MS10, IDS>, (unsigned)((p.n_streams + SYN_WARPS - 1) / SYN_WARPS), SYN_WARPS * 32,
                        synth_warp_smem_bytes(NF, 1), p, dep);
    }
};
}  // namespace

cudaError_t prepare_synth(const DecoderState& st) {
    PrepareSynth ps;
    if (!dispatch_frame_geo(st.cfg.nf, st.cfg.n_ms == LC3B_10MS, ps)) return cudaErrorInvalidValue;
    if (ps.e != cudaSuccess) return ps.e;
    const int lb = (int)(ltpf_warp_bytes(st.cfg) * SYN_WARPS);
    const cudaError_t e = cudaFuncSetAttribute(ltpf_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, lb);
    return e != cudaSuccess ? e : cudaFuncSetAttribute(ltpf_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, lb);
}

// Adds the synthesis kernel (after node `dep`, -1 = none) and the post-filter kernel behind it; returns the last node.
int plan_synth(LaunchPlan& plan, const DecoderState& st, int16_t* pcm_out, size_t pcm_stride, int dep, int base, int count,
               const int32_t* ids) {
    SynthParams p;
    memset(&p, 0, sizeof(p));
    p.cfg = st.dcfg;
    p.win = st.win;
    p.dtw = st.dtw;
    p.ftw = st.ftw;
    // a sub-batch: every per-stream pointer moved to its first stream, or with an id list only the rows (see entropy_params)
    const size_t b = (size_t)base, sb = ids ? 0 : b;
    const int n = count < 0 ? st.n_streams : count;
    p.hist_len = (st.cfg.n_ms == LC3B_10MS ? 2 : 3) * st.cfg.nf;
    p.spec = st.spec + sb * st.cfg.ne;
    p.ola = st.ola + sb * (size_t)(st.cfg.nf - st.cfg.z);
    p.ltpf_y = st.ltpf_y + sb * (size_t)p.hist_len;
    p.ltpf_xtail = st.ltpf_xtail + sb * XTAIL_FLOATS;
    p.ltpf_x = st.ltpf_x + sb * (size_t)st.cfg.nf;
    p.side = st.side + sb * SIDE_WORDS;
    p.sstate = st.sstate + sb * SS_WORDS;
    p.pcm_out = pcm_out + b * pcm_stride;
    p.ids = ids ? ids + b : nullptr;
    p.pcm_stride = pcm_stride;
    p.n_streams = n;
    p.slot_streams = st.n_streams;
    p.pcm_pairs = (((uintptr_t)p.pcm_out & 3) == 0 && (pcm_stride & 1) == 0) ? 1 : 0;
    // ltpf_kernel: one warp per stream while that keeps the grid small, else a warp walks a group of streams
    int group = 1;
    while (group < 32 && n / group > 16384) group *= 2;
    p.group = group;
    const size_t lw = ltpf_warp_bytes(st.cfg);
    p.smem_per_warp = (int)lw;
    p.no_ltpf = st.no_ltpf;
    // which synthesis kernel (lc3b_decoder_set_synth_mode): 0 = by launch size (default), 1 = one frame per warp always
    PlanSynth ps{plan, p, dep, -1, st.sm_count > 0 ? st.sm_count : 148, st.synth_mode == 1};
    if (!dispatch_frame_geo(st.cfg.nf, st.cfg.n_ms == LC3B_10MS, ps)) return -1;
    if (st.no_ltpf) return ps.node;                           // the post filter can never be active: nothing to launch
    const int n_warps = (n + group - 1) / group;
    return plan.add(ids ? ltpf_kernel<true> : ltpf_kernel<false>, (unsigned)((n_warps + SYN_WARPS - 1) / SYN_WARPS), SYN_WARPS * 32,
                    lw * SYN_WARPS, p, ps.node);
}

}  // namespace lc3b
