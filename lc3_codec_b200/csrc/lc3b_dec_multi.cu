// lc3b engine: time-parallel decode - many consecutive frames of many streams in ONE call (SURVEY.md 8f-1).
//
// The reference decodes a file frame by frame (examples/decode.rs:85-123); with few channels that leaves a GPU idle.
// Of the decoder's state only three things really run along time:
//   * overlap-add needs the previous frame's windowed tail            (modified_dct.rs:138-151)  -> one add
//   * concealment needs the last good spectrum, a fading factor and an LCG seed (packet_loss_concealment.rs:63-85)
//                                                                     -> a scan over the frames' ok flags
//   * the LTPF is an IIR across frame boundaries, but only while it is active (long_term_post_filter.rs:252)
// A call lists rows in a row table (lc3b_common.cuh): row i advances handle stream row_i by count_i consecutive frames,
// units off_i .. off_i + count_i - 1.  lc3b_decode_stream_frames_subset sends its table; lc3b_decode_stream_frames is the
// identity table of S rows of F frames, which unit_rows_kernel writes on the device.  The units run independently through
// the expensive stages and the time axis is touched only where it must be:
//   1. entropy_kernel + dequant_kernel over the units (the unchanged kernels; spectrum to a per-unit slot)
//   2. unit_rows_kernel     warp per row: unit_row[v], the state row of each unit's row (stages 3 and 4 read it)
//      plc_scan_kernel      warp per row: walks the ok flags, assigns each concealed unit its source spectrum,
//                           alpha and seed (the LCG is jumped ne steps at a time), updates the handle's PLC scalars
//   3. imdct_multi_kernel   warp per unit: concealment scramble, DCT-IV (same FFT as kernel 2), window -> head / tail
//   4. ola_multi_kernel     warp per unit: x_hat = head + previous unit's tail, PCM of every frame
//   5. ltpf_multi_kernel    warp per row: replays the post filter over the spans where it is (or just was) active,
//                           overwriting those frames' PCM; then leaves the handle's per-stream state (overlap memory,
//                           LTPF ring, last good spectrum) exactly as count_i frame-by-frame calls would have
// Arithmetic is the frame-by-frame path's, operation for operation, so both paths produce identical PCM.
#include "lc3b_common.cuh"
#include "lc3b_imdct.cuh"
#include "lc3b_plan.cuh"
#include "lc3b_math.cuh"
#include "lc3b_synth.cuh"

namespace lc3b {

struct MultiLayout { size_t rows, spec, xq, handoff, gband, tns_list, side, head, tail, xhat, last_good, unit_row, total; };

// V units of S rows: the row table at the front (where RowTable::send puts it) and unit_row[V] at the end
static MultiLayout multi_layout(const lc3b_config& c, int S, size_t V) {
    MultiLayout L;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = (off + bytes + 255) & ~(size_t)255; return o; };
    L.rows = take(sizeof(int32_t) * RT_WORDS * S);
    const size_t nblk = ((V + 127) / 128) * 4;                    // 32-stream blocks, whole entropy CTAs
    L.spec = take(sizeof(float) * V * c.ne);
    L.xq = take(sizeof(int32_t) * nblk * c.ne * 32);
    L.handoff = take(sizeof(int32_t) * nblk * 32 * HO_WORDS);
    L.gband = take(sizeof(float) * nblk * 32 * 64);             // small unit counts take the warp-per-frame dequantisation
    L.tns_list = take(sizeof(int32_t) * (2 + nblk * 32));
    L.side = take(sizeof(int32_t) * V * SIDE_WORDS);
    L.head = take(sizeof(float) * V * c.nf);
    L.tail = take(sizeof(float) * V * (c.nf - c.z));
    L.xhat = take(sizeof(float) * V * c.nf);
    L.last_good = take(sizeof(int32_t) * S);
    L.unit_row = take(sizeof(int32_t) * V);
    L.total = off;
    return L;
}

size_t multi_scratch_bytes(const DecoderState& st, int n_rows, long long total) {
    return multi_layout(st.cfg, n_rows, (size_t)total).total;
}

struct MultiParams {
    const DevConfig* cfg;
    const float* win;
    const float2* dtw;
    const float2* ftw;
    int S;                // the handle's streams (stride between its two spectrum slots)
    int n_rows, V;        // rows of the row table, units
    const int32_t* rows;  // row table (lc3b_common.cuh)
    const int32_t* unit_row;   // [V] the state row of each unit's row, ~row for a row's first unit
    // per-unit scratch
    const float* spec_v;
    int32_t* side_v;
    float* head;
    float* tail;
    float* xhat;
    int32_t* last_good;   // [rows]
    // the handle's per-stream state
    float* spec;
    float* ola;
    float* ltpf_y;
    float* ltpf_xtail;
    int32_t* sstate;
    int16_t* pcm_out;
    int hist_len;
    int smem_per_warp;    // ltpf_multi_kernel, bytes
};

constexpr int MW = 4;     // warps per CTA in the warp-per-unit kernels

// ---------------------------------------------------------------- 2. concealment bookkeeping along time
// One warp per row; the ok flags are fetched 32 frames at a time so that the walk along time is not one dependent
// global load per frame.  Every lane tracks the same running state; lane j writes frame j's record.
__global__ void __launch_bounds__(MW * 32) plc_scan_kernel(MultiParams p) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int r = blockIdx.x * MW + wid;
    if (r >= p.n_rows) return;
    const RowSpan rs = row_span(p.rows, r);
    const int s = rs.row, F = rs.count, v0 = rs.off;
    const int ne = p.cfg->ne;
    int32_t* ss = p.sstate + (size_t)s * SS_WORDS;
    int lost = ss[SS_PLC_LOST];
    float alpha = u2f((uint32_t)ss[SS_PLC_ALPHA]);
    uint32_t seed = (uint32_t)ss[SS_PLC_SEED];
    __syncwarp();
    const PlcJump jump = plc_lcg_jump(ne);                         // a concealed frame takes ne steps of the LCG
    int last = -1;
    for (int f0 = 0; f0 < F; f0 += 32) {
        const int f = f0 + lane;
        const int v = v0 + f;
        int32_t* sd = p.side_v + (size_t)v * SIDE_WORDS;
        const bool in = f < F;
        const bool ok = in && sd[SD_OK] != 0;
        const uint32_t okm = __ballot_sync(0xffffffffu, ok), inm = __ballot_sync(0xffffffffu, in);
        if (okm == inm) {                                          // the usual chunk: every frame decoded
            if (in) sd[SD_SRC] = -2;
            lost = 0;
            alpha = 1.0f;
            last = v0 + f0 + (31 - __clz(inm));
            continue;
        }
        const int cnt = __popc(inm);
        for (int j = 0; j < cnt; j++) {
            if ((okm >> j) & 1u) {
                lost = 0;
                alpha = 1.0f;
                last = v0 + f0 + j;
                if (lane == j) sd[SD_SRC] = -2;
            } else {
                alpha = plc_fade(alpha, lost);
                if (lane == j) {
                    sd[SD_SRC] = last;
                    sd[SD_PLC_ALPHA] = (int32_t)f2u(alpha);
                    sd[SD_PLC_SEED] = (int32_t)seed;
                }
                seed = jump.step(seed);
                lost++;
            }
        }
    }
    if (lane == 0) {
        ss[SS_PLC_LOST] = lost;
        ss[SS_PLC_ALPHA] = (int32_t)f2u(alpha);
        ss[SS_PLC_SEED] = (int32_t)seed;
        p.last_good[r] = last;
    }
}

// ---------------------------------------------------------------- 3. spectrum -> windowed time signal, per unit
template <int NF, bool MS10>
__global__ void __launch_bounds__(MW * 32) imdct_multi_kernel(MultiParams p) {
    using G = FrameGeo<NF, MS10>;
    constexpr int NE = G::NE, Z = G::Z, NP = G::NP, NPT = G::NPT;
    extern __shared__ __align__(16) uint8_t smem[];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const long long v = (long long)blockIdx.x * MW + wid;
    if (v >= (long long)p.V) return;
    float* P = (float*)smem + (size_t)wid * 2 * NF;
    float* Q = P + NF;

    const int32_t* sd = p.side_v + (size_t)v * SIDE_WORDS;
    const int src = sd[SD_SRC];
    const float* sp;
    if (src == -2) sp = p.spec_v + (size_t)v * NE;
    else if (src >= 0) sp = p.spec_v + (size_t)src * NE;
    else {                                                        // last good of earlier calls
        const int sr = unit_state_row(p.unit_row[v]);
        sp = p.spec + ((size_t)p.sstate[(size_t)sr * SS_WORDS + SS_SLOT] * p.S + sr) * NE;
    }
    if (src == -2) {
#pragma unroll
        for (int k0 = 0; k0 < NF / 4; k0 += 32) {
            const int k4 = k0 + lane;
            if (k0 + 32 <= NF / 4 || k4 < NF / 4)
                ((float4*)P)[k4] = 4 * k4 < NE ? ((const float4*)sp)[k4] : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        }
    } else {                                                      // concealed: the source spectrum, scrambled
        plc_scramble<NF, NE>(P, sp, u2f((uint32_t)sd[SD_PLC_ALPHA]), (uint32_t)sd[SD_PLC_SEED], lane);
    }
    __syncwarp();
    const float* D = dct_iv_warp<NF>(P, Q, p.dtw, p.ftw, lane);
    float hd[2 * NP], tl[2 * NPT];
    imdct_unfold<NF, MS10>(D, p.win, lane, hd, tl);
    float2* head = (float2*)(p.head + (size_t)v * NF);
    float2* tail = (float2*)(p.tail + (size_t)v * (NF - Z));
#pragma unroll
    for (int j = 0; j < NP; j++)
        if (64 * j + 64 <= NF || 64 * j + 2 * lane < NF) head[32 * j + lane] = make_float2(hd[2 * j], hd[2 * j + 1]);
#pragma unroll
    for (int j = 0; j < NPT; j++)
        if (64 * j + 64 <= NF - Z || 64 * j + 2 * lane < NF - Z) tail[32 * j + lane] = make_float2(tl[2 * j], tl[2 * j + 1]);
}

// ---------------------------------------------------------------- 4. overlap-add across units, PCM
__global__ void __launch_bounds__(MW * 32) ola_multi_kernel(MultiParams p) {
    const DevConfig& c = *p.cfg;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const long long v = (long long)blockIdx.x * MW + wid;
    if (v >= (long long)p.V) return;
    const int nf = c.nf, z = c.z;
    const int u = __ldg(p.unit_row + v);                           // >= 0: not the first frame of its row, the previous unit's tail
    const float* head = p.head + (size_t)v * nf;
    const float* prev = u >= 0 ? p.tail + (size_t)(v - 1) * (nf - z) : p.ola + (size_t)~u * (nf - z);
    float* xhat = p.xhat + (size_t)v * nf;
    int16_t* out = p.pcm_out + (size_t)v * nf;
    // read-only loads: the compiler may then issue all of a lane's loads before its stores to xhat and out, which it would
    // otherwise have to assume alias them (a unit's row costs this kernel one more load latency than v / F did)
    for (int n = lane; n < nf; n += 32) {
        float o = __ldg(head + n);
        if (n < nf - z) o = xa(__ldg(prev + n), o);
        xhat[n] = o;
        out[n] = (int16_t)round_pcm_i32(o);
    }
}

// ---------------------------------------------------------------- 5. LTPF over its active spans + state hand-back
// One warp per CTA: the row is then blockIdx.x, which ptxas knows to be the same for the whole warp, and so are the
// row's entry and the bound of the walk.  With four warps per CTA they are per-thread values to it: the walk's control
// flow leaves the uniform datapath and the kernel ran 5 % slower on bench.py --workload file16.  The minimum of 32 CTAs
// per SM holds it to 64 registers (and 32 warps per SM); without it ptxas takes 72 and still spills a little.
__global__ void __launch_bounds__(32, 32) ltpf_multi_kernel(MultiParams p) {
    extern __shared__ __align__(16) uint8_t smem[];
    const DevConfig& c = *p.cfg;
    const int lane = threadIdx.x;
    const int r = blockIdx.x;
    const RowSpan rs = row_span(p.rows, r);
    const int s = rs.row;
    const LtpfGeo g = ltpf_geo(c, p.hist_len);
    const int nf = g.nf, ne = c.ne, z = c.z, F = rs.count, blocks = g.blocks;
    float* Y = (float*)smem;                                       // see ltpf_warp_bytes
    float* X = Y + p.hist_len;
    float* xt = X + nf;
    float* scratch = xt + 16;
    int32_t* ss = p.sstate + (size_t)s * SS_WORDS;
    float* yhist = p.ltpf_y + (size_t)s * p.hist_len;
    float* xtail = p.ltpf_xtail + (size_t)s * XTAIL_FLOATS;      // [blocks][16], slot = ring block of the frame it closes
    const int blk0 = ss[SS_LTPF_BLK];
    LtpfPar prev = ltpf_load_prev(ss);
    const int slot = ss[SS_SLOT];
    __syncwarp();
    for (int n = lane; n < p.hist_len; n += 32) Y[n] = yhist[n];
    __syncwarp();
    bool span1 = false, span2 = false, span3 = false;              // were frames f-1 / f-2 / f-3 filtered by this kernel
    const size_t v0 = (size_t)rs.off;
    uint32_t actm = 0;                                             // LTPF-active flags of the current 32-frame chunk
    for (int f = 0; f < F; f++) {
        if ((f & 31) == 0) {                                       // fetch 32 frames' flags at once; skip idle chunks
            const int fl = f + lane;
            actm = __ballot_sync(0xffffffffu, fl < F && p.side_v[(v0 + fl) * SIDE_WORDS + SD_LTPF_ACTIVE] != 0);
            if (actm == 0 && !prev.active) {
                span1 = span2 = span3 = false;
                prev = LtpfPar{};
                f += 31;
                continue;
            }
        }
        const size_t v = v0 + f;
        const LtpfPar cur = ltpf_params(c, p.side_v + v * SIDE_WORDS);
        const bool in_span = cur.active || prev.active;
        if (in_span) {
            const int blk = ((blk0 + f) % blocks) * nf;
            // history this frame may read: frames f-1 .. f-blocks (the oldest one sits in the block this frame is about
            // to overwrite: the ring is circular and long pitch lags reach into it); refill the ones this kernel skipped
            for (int j = 1; j <= blocks; j++) {
                const int g = f - j;
                const bool have = j == 1 ? span1 : j == 2 ? span2 : span3;
                if (g >= 0 && !have) {
                    const float* src = p.xhat + (v0 + g) * nf;
                    float* dst = Y + ((blk0 + g) % blocks) * nf;
                    for (int n = lane; n < nf; n += 32) dst[n] = src[n];
                }
            }
            const float* xh = p.xhat + v * nf;
            for (int n = lane; n < nf; n += 32) X[n] = xh[n];
            if (lane < 16) xt[lane] = f > 0 ? p.xhat[(v - 1) * nf + nf - 16 + lane] : xtail[((blk0 + blocks - 1) % blocks) * 16 + lane];
            __syncwarp();
            ltpf_filter_frame(c, g, Y, X, xt, scratch, blk, cur, prev, lane);
            int16_t* out = p.pcm_out + v * nf;
            for (int n = lane; n < nf; n += 32) out[n] = (int16_t)round_pcm_i32(Y[blk + n]);
            __syncwarp();
        }
        span3 = span2;
        span2 = span1;
        span1 = in_span;
        prev = cur;
    }
    if (F == 0) return;
    // ---- hand the per-stream state back as F frame-by-frame calls would have left it
    for (int j = 0; j < blocks; j++) {                             // LTPF ring: the last `blocks` frames' output
        const int g = F - 1 - j;
        if (g < 0) break;
        const int bo = ((blk0 + g) % blocks) * nf;
        const bool have = j == 0 ? span1 : j == 1 ? span2 : span3;
        const float* src = have ? Y + bo : p.xhat + (v0 + g) * nf;
        for (int n = lane; n < nf; n += 32) yhist[bo + n] = src[n];
    }
    if (lane < 16) xtail[((blk0 + F - 1) % blocks) * 16 + lane] = p.xhat[(v0 + F - 1) * nf + nf - 16 + lane];
    {
        const float* t = p.tail + (v0 + F - 1) * (nf - z);
        float* ola = p.ola + (size_t)s * (nf - z);
        for (int n = lane; n < nf - z; n += 32) ola[n] = t[n];
    }
    const int lg = p.last_good[r];
    if (lg >= 0) {                                                 // PacketLossConcealment::save of the last good frame
        const float* src = p.spec_v + (size_t)lg * ne;
        float* dst = p.spec + ((size_t)(slot ^ 1) * p.S + s) * ne;
        for (int k = lane; k < ne; k += 32) dst[k] = src[k];
    }
    if (lane == 0) {
        ltpf_store_prev(ss, prev);
        ss[SS_LTPF_BLK] = (blk0 + F) % blocks;
        if (lg >= 0) ss[SS_SLOT] = slot ^ 1;
    }
}

// ---------------------------------------------------------------- each unit's row, for stages 3 and 4
constexpr int UR_WARPS = 8;   // warps per CTA of unit_rows_kernel: a dense call of many short rows is thousands of CTAs

struct UnitRowsParams {
    int32_t* rows;        // row table; written here for a dense call
    int32_t* unit_row;
    int n_rows;
    int dense_frames;     // > 0: a dense call, row r is stream r with dense_frames frames from unit r * dense_frames
};

__global__ void __launch_bounds__(UR_WARPS * 32) unit_rows_kernel(UnitRowsParams p) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int r = blockIdx.x * UR_WARPS + wid;
    if (r >= p.n_rows) return;
    RowSpan rs;
    if (p.dense_frames > 0) {
        rs = RowSpan{r, r * p.dense_frames, p.dense_frames};
        if (lane == 0) {
            int32_t* w = p.rows + RT_WORDS * r;
            w[RT_ROW] = rs.row;
            w[RT_OFF] = rs.off;
            w[RT_COUNT] = rs.count;
        }
    } else {
        rs = row_span(p.rows, r);
    }
    for (int f = lane; f < rs.count; f += 32) p.unit_row[(size_t)rs.off + f] = f ? rs.row : ~rs.row;
}

void plan_unit_rows(LaunchPlan& plan, int32_t* rows, int n_live, int dense_frames, int32_t* unit_row) {
    const UnitRowsParams p{rows, unit_row, n_live, dense_frames};
    plan.add(unit_rows_kernel, (unsigned)((n_live + UR_WARPS - 1) / UR_WARPS), UR_WARPS * 32, 0, p);
}

namespace {
struct PrepareImdct {
    cudaError_t e = cudaSuccess;
    template <int NF, bool MS10> void operator()() {
        e = cudaFuncSetAttribute(imdct_multi_kernel<NF, MS10>, cudaFuncAttributeMaxDynamicSharedMemorySize, MW * 2 * NF * 4);
    }
};
struct PlanImdct {
    LaunchPlan& plan;
    const MultiParams& p;
    unsigned grid;
    template <int NF, bool MS10> void operator()() { plan.add(imdct_multi_kernel<NF, MS10>, grid, MW * 32, MW * 2 * NF * 4, p); }
};
}  // namespace

cudaError_t prepare_multi(const DecoderState& st) {
    cudaError_t e = cudaFuncSetAttribute(ltpf_multi_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ltpf_warp_bytes(st.cfg));
    if (e == cudaSuccess) {
        PrepareImdct pi;
        if (!dispatch_frame_geo(st.cfg.nf, st.cfg.n_ms == LC3B_10MS, pi)) return cudaErrorInvalidValue;
        e = pi.e;
    }
    return e;
}

cudaError_t launch_decode_multi(const DecoderState& st, const uint8_t* frames, const int32_t* frame_nbytes, int nbytes,
                                size_t frame_stride, int n_rows, int n_live, long long V, int dense_frames, int16_t* pcm_out,
                                int32_t* status_out, void* scratch, cudaStream_t stream, PlanLanes* lanes) {
    if (V <= 0) return cudaSuccess;
    const MultiLayout L = multi_layout(st.cfg, n_rows, (size_t)V);
    uint8_t* base = (uint8_t*)scratch;
    // 1. entropy decode of all units with the unchanged kernel: a view of the handle with V virtual streams
    DecoderState vs = st;
    vs.n_streams = (int)V;
    vs.spec = (float*)(base + L.spec);
    vs.xq = (int32_t*)(base + L.xq);
    vs.handoff = (int32_t*)(base + L.handoff);
    vs.gband = (float*)(base + L.gband);
    vs.tns_list = (int32_t*)(base + L.tns_list);
    vs.nsym_prev = nullptr;                                       // units of one call are not consecutive frames of a stream slot
    vs.side = (int32_t*)(base + L.side);
    vs.fixed_slot = 0;
    vs.trace = nullptr;
    vs.trace_x = nullptr;
    cudaError_t e = cudaMemsetAsync(vs.tns_list, 0, 2 * sizeof(int32_t), stream);   // caller-owned scratch: the list starts empty
    if (e == cudaSuccess) {
        // large calls: the units as four independent sub-batches whose kernels overlap (run_decode in lc3b_api.cu)
        LaunchPlan plan;
        const int n = vs.n_streams;
        const int k_sub = (lanes && n >= decode_split_min_streams() && !use_dequant_warp(n, vs.dequant_mode)) ? PLAN_MAX_LANES : 1;
        int part = ((n + k_sub - 1) / k_sub + 127) & ~127;
        if (k_sub == 1) part = n;
        for (int k = 0, b = 0; k < k_sub && b < n; k++, b += part) {
            plan.lane = k;
            plan_entropy(plan, vs, frames, frame_nbytes, nbytes, frame_stride, status_out, 3, b, k_sub == 1 ? -1 : (n - b < part ? n - b : part), -1);
        }
        e = plan_launch_direct(plan, stream, lanes);
    }
    if (e != cudaSuccess) return e;
    int32_t* rows = (int32_t*)(base + L.rows);
    int32_t* unit_row = (int32_t*)(base + L.unit_row);
    MultiParams p;
    memset(&p, 0, sizeof(p));
    p.cfg = st.dcfg; p.win = st.win; p.dtw = st.dtw; p.ftw = st.ftw;
    p.S = st.n_streams;
    p.n_rows = n_live; p.V = (int)V;
    p.rows = rows;
    p.unit_row = unit_row;
    p.spec_v = vs.spec; p.side_v = vs.side;
    p.head = (float*)(base + L.head); p.tail = (float*)(base + L.tail); p.xhat = (float*)(base + L.xhat);
    p.last_good = (int32_t*)(base + L.last_good);
    p.spec = st.spec; p.ola = st.ola; p.ltpf_y = st.ltpf_y; p.ltpf_xtail = st.ltpf_xtail; p.sstate = st.sstate;
    p.pcm_out = pcm_out;
    p.hist_len = (st.cfg.n_ms == LC3B_10MS ? 2 : 3) * st.cfg.nf;
    p.smem_per_warp = (int)ltpf_warp_bytes(st.cfg);
    // 2-5. a second plan on the caller's stream: plan_launch_direct joins the entropy plan's lanes back into the caller's
    // stream only at the end of that plan, so lane-0 nodes added to it would not wait for lanes 1-3
    LaunchPlan tail;
    const unsigned grid_s = (unsigned)((n_live + MW - 1) / MW), grid_v = (unsigned)((V + MW - 1) / MW);
    plan_unit_rows(tail, rows, n_live, dense_frames, unit_row);
    tail.add(plc_scan_kernel, grid_s, MW * 32, 0, p);
    PlanImdct pi{tail, p, grid_v};
    if (!dispatch_frame_geo(st.cfg.nf, st.cfg.n_ms == LC3B_10MS, pi)) return cudaErrorInvalidValue;
    tail.add(ola_multi_kernel, grid_v, MW * 32, 0, p);
    tail.add(ltpf_multi_kernel, (unsigned)n_live, 32, (size_t)p.smem_per_warp, p);
    return plan_launch_direct(tail, stream);
}

}  // namespace lc3b
