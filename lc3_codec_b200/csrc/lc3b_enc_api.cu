// lc3b engine: encoder half of the C ABI (include/lc3b.h) - configuration tables, workspace carving, launch sequencing.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <new>

#include "lc3b_enc_common.cuh"
#include "lc3b_handles.cuh"
#include "lc3b_math.cuh"
#include "lc3_tables.h"

namespace lc3b {

// CUDA failures of the encoder land in the same thread-local slot as the decoder's (lc3b_last_cuda_error)
#define CU(x) LC3B_CU(x)

struct EncLayout {
    size_t ecfg, win, dtw, ftw, perm, thist, xs_hist, x12, x6, estate, xf, e_b, ehand, xq, qhand, lsbs, bs_scratch, stage_in,
        stage_out, ids, total;
};

static size_t take(size_t& off, size_t bytes) {
    size_t o = off;
    off += (bytes + 255) & ~(size_t)255;
    return o;
}

__host__ __device__ static int x12_len_of(const lc3b_config& c) { return (c.n_ms == LC3B_10MS ? 128 + 24 : 96 + 44) + 232; }

static EncLayout make_enc_layout(const lc3b_config& c, int n_streams, int max_nbytes) {
    EncLayout L;
    size_t off = 0;
    const size_t ns = (size_t)n_streams;
    L.ecfg = take(off, sizeof(EncConfig));
    L.win = take(off, sizeof(float) * 2 * c.nf);
    L.dtw = take(off, sizeof(float2) * (c.nf / 2));
    L.ftw = take(off, sizeof(float2) * (c.nf / 2));
    L.perm = take(off, sizeof(int32_t) * (c.nf / 2));
    L.thist = take(off, sizeof(int16_t) * ns * (c.nf - c.z));
    L.xs_hist = take(off, sizeof(int16_t) * ns * 64);
    L.x12 = take(off, sizeof(float) * ns * x12_len_of(c));
    L.x6 = take(off, sizeof(float) * ns * 178);
    L.estate = take(off, sizeof(int32_t) * ns * ES_WORDS);
    L.xf = take(off, sizeof(float) * ns * c.ne);
    L.e_b = take(off, sizeof(float) * ns * 64);
    L.ehand = take(off, sizeof(int32_t) * ns * EH_WORDS);
    L.xq = take(off, sizeof(int16_t) * ns * c.ne);
    L.qhand = take(off, sizeof(int32_t) * ns * QH_WORDS);
    L.lsbs = take(off, ns * 2 * c.ne);
    L.bs_scratch = take(off, ns * sizeof(uint32_t) * (size_t)enc_bitstream_scratch_words(c.ne, max_nbytes));
    L.stage_in = take(off, sizeof(int16_t) * ns * c.nf * 2);   // double-buffered for the pipelined host path
    L.stage_out = take(off, ns * (size_t)max_nbytes);
    L.ids = take(off, sizeof(int32_t) * ns);                    // id list of a subset call (lc3b_encode_frames_subset)
    L.total = off;
    return L;
}

__global__ void enc_init_tables_kernel(const EncConfig* cfg, float* win) {
    const int nf = cfg->nf;
    const float* w;
    if (cfg->n_ms == LC3B_7P5MS) {
        w = nf == 60 ? LC3T_W_N60_7P5MS : nf == 120 ? LC3T_W_N120_7P5MS : nf == 180 ? LC3T_W_N180_7P5MS
            : nf == 240 ? LC3T_W_N240_7P5MS : LC3T_W_N360_7P5MS;
    } else {
        w = nf == 80 ? LC3T_W_N80_10MS : nf == 160 ? LC3T_W_N160_10MS : nf == 240 ? LC3T_W_N240_10MS
            : nf == 320 ? LC3T_W_N320_10MS : LC3T_W_N480_10MS;
    }
    for (int m = threadIdx.x; m < 2 * nf; m += blockDim.x) win[m] = w[m];
}

__global__ void enc_init_band_kernel(EncConfig* cfg) {
    const uint16_t* bi;
    if (cfg->n_ms == LC3B_7P5MS) {
        bi = cfg->fs_ind == 0 ? LC3T_I_8000_7P5MS : cfg->fs_ind == 1 ? LC3T_I_16000_7P5MS
             : cfg->fs_ind == 2 ? LC3T_I_24000_7P5MS : cfg->fs_ind == 3 ? LC3T_I_32000_7P5MS : LC3T_I_48000_7P5MS;
    } else {
        bi = cfg->fs_ind == 0 ? LC3T_I_8000_10MS : cfg->fs_ind == 1 ? LC3T_I_16000_10MS
             : cfg->fs_ind == 2 ? LC3T_I_24000_10MS : cfg->fs_ind == 3 ? LC3T_I_32000_10MS : LC3T_I_48000_10MS;
    }
    for (int b = threadIdx.x; b < 65; b += blockDim.x) cfg->band_idx[b] = b <= cfg->nb ? bi[b] : cfg->ne;
    {
        const int up = cfg->up, kq = 120 / up;
        for (int i = threadIdx.x; i < 240; i += blockDim.x) {
            const int r = i / (2 * kq), j = i - r * (2 * kq);
            const int index_h = up * (j - kq + 1) - r;
            cfg->resamp_ph[i] = (index_h > -120 && index_h < 120) ? LC3T_TAB_RESAMP_FILTER[119 + index_h] : 0.0f;
        }
    }
    for (int k = threadIdx.x; k < 400; k += blockDim.x) {
        int band = 255;
        for (int b = 0; b < cfg->nb; b++) if (k >= bi[b] && k < bi[b + 1]) band = b;
        cfg->band_of[k] = (uint8_t)band;
        cfg->band_width_of[k] = band == 255 ? 0.0f : (float)(bi[band + 1] - bi[band]);
    }
}

// The state a stream starts from.  ids == nullptr: every stream, whose rows lc3b_encoder_init has just zeroed with the
// rest of the workspace; otherwise the n listed streams (lc3b_encoder_reset_streams), whose persistent rows are zeroed
// here first - one warp per stream.
__global__ void enc_init_streams_kernel(EncoderState st, const int32_t* ids, int n) {
    const int lane = threadIdx.x & 31;
    const int i = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    if (i >= n) return;
    const int s = ids ? ids[i] : i;
    if (ids) {
        const int nz = st.cfg.nf - st.cfg.z, x12_len = x12_len_of(st.cfg);
        for (int k = lane; k < nz; k += 32) st.thist[(size_t)s * nz + k] = 0;
        for (int k = lane; k < 64; k += 32) st.xs_hist[(size_t)s * 64 + k] = 0;
        for (int k = lane; k < x12_len; k += 32) st.x12[(size_t)s * x12_len + k] = 0.0f;
        for (int k = lane; k < 178; k += 32) st.x6[(size_t)s * 178 + k] = 0.0f;
    }
    if (lane != 0) return;
    int32_t* es = st.estate + (size_t)s * ES_WORDS;
    for (int k = 0; k < ES_WORDS; k++) es[k] = 0;
    es[ES_ATT_POS_LAST] = -1;      // attack_detector.rs:38
    es[ES_T_PREV] = 17;            // long_term_post_filter.rs:85 (K_MIN)
}

static cudaError_t launch_enc_init_streams(const EncoderState& st, const int32_t* ids, int n, cudaStream_t stream) {
    enc_init_streams_kernel<<<(unsigned)((n + 7) / 8), 256, 0, stream>>>(st, ids, n);
    return cudaGetLastError();
}

// host-side construction of everything that does not need the device tables
static void fill_enc_config(const lc3b_config& c, EncConfig* d, float2* dtw, float2* ftw, int32_t* perm) {
    memset(d, 0, sizeof(*d));
    d->fs_ind = c.fs_ind; d->fs = c.fs; d->ne = c.ne; d->nb = c.nb; d->nf = c.nf; d->z = c.z; d->n_ms = c.n_ms;
    const int N = c.nf / 2;
    d->n_fft = N;
    {   // kf_factor, kissfft.rs:47-76
        int p = 4, rem = N, lv = 0, fs = 1;
        const float floor_sqrt = floorf(sqrtf((float)N));
        for (;;) {
            while (rem % p != 0) {
                if (p == 4) p = 2;
                else if (p == 2) p = 3;
                else p += 2;
                if ((float)p > floor_sqrt) p = rem;
            }
            rem /= p;
            d->fac_p[lv] = p;
            d->fac_m[lv] = rem;
            d->fac_stride[lv] = fs;
            fs *= p;
            lv++;
            if (rem <= 1) break;
        }
        d->n_levels = lv;
        for (int o = 0; o < N; o++) {          // leaf permutation: o = sum d_i * m_i  ->  in = sum d_i * fstride_i
            int r = o, in = 0;
            for (int i = 0; i < lv; i++) {
                const int di = r / d->fac_m[i];
                r -= di * d->fac_m[i];
                in += di * d->fac_stride[i];
            }
            perm[o] = in;
        }
    }
    for (int i = 0; i < N; i++) {              // dct_iv.rs:30-35, kissfft.rs:19-29: f64 then narrowed
        const double t = -M_PI * (double)(8 * i + 1) / (8.0 * (double)N * 2.0);
        dtw[i] = make_float2((float)cos(t), (float)sin(t));
        const double ph = -2.0 * M_PI * (double)i / (double)N;
        ftw[i] = make_float2((float)cos(ph), (float)sin(ph));
    }
    if (c.n_ms == LC3B_10MS) { d->len12p8 = 128; d->len6p4 = 64; d->delay = 24; d->att_num_ds = 160; d->att_num_blocks = 4; d->att_pos_limit = 2; }
    else { d->len12p8 = 96; d->len6p4 = 48; d->delay = 44; d->att_num_ds = 120; d->att_num_blocks = 3; d->att_pos_limit = 1; }
    int ext;
    switch (c.fs) {
        case 8000: d->up = 24; d->resamp_fac = 0.5f; ext = 10; break;
        case 16000: d->up = 12; d->resamp_fac = 1.0f; ext = 20; break;
        case 24000: d->up = 8; d->resamp_fac = 1.0f; ext = 30; break;
        case 32000: d->up = 6; d->resamp_fac = 1.0f; ext = 40; break;
        default: d->up = 4; d->resamp_fac = 1.0f; ext = 60; break;
    }
    d->x_s_ext_len = ext + c.nf;
    d->x12_len = x12_len_of(c);
    const float step = (float)M_PI / 17.0f;                                    // temporal_noise_shaping.rs:268
    for (int k = 0; k < 17; k++) d->tns_sin[k] = (float)sin((double)(step * ((float)k - 8.0f)));
    for (int k = 0; k < 400; k++) d->gg_table[k] = powf_msun(10.0f, (float)(k - 245) / 28.0f);
    static const int G_TILT[5] = {14, 18, 22, 26, 30};                          // spectral_noise_shaping.rs:51-57
    const float exponent = (float)G_TILT[c.fs_ind] / 630.0f;
    for (int b = 0; b < 64; b++) d->pre_emph[b] = powf_msun(10.0f, (float)b * exponent);
}

}  // namespace lc3b

using namespace lc3b;

struct lc3b_encoder {
    EncoderState st{};
    int stage_mask = 63;
    int graph_mode = 0;                 // 0 = one launch per kernel, 1 = one cached CUDA graph per call (lc3b_plan.cuh)
    GraphCache graphs;
    IdList id_list;                     // subset calls and resets (lc3b_encode_frames_subset, lc3b_encoder_reset_streams)
    RowTable row_table;                 // ragged time-parallel calls (lc3b_encode_stream_frames_subset)
    // optional pipelining of the host entry point: PCM arrives on an internal copy stream into a double-buffered
    // staging area, so the upload of call i+1 overlaps the kernels of call i
    int pipelined = 0, buf = 0;
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t h2d_done[2] = {nullptr, nullptr}, consumed[2] = {nullptr, nullptr};
    bool consumed_valid[2] = {false, false};
};

// the kernels of one encode_frame per stream (ids == nullptr) or per row of a subset call (n rows, row u = stream ids[u],
// ids in device memory) as a plan: stage mask bits 0-1 analysis, bits 2-5 quantisation / bitstream
static cudaError_t run_encode(lc3b_encoder* h, const int16_t* pcm, size_t pcm_stride, uint8_t* frames_out, int nbytes,
                              size_t frame_stride, int mask, cudaStream_t stream, const int32_t* ids = nullptr, int n = 0) {
    LaunchPlan plan;
    EncoderState v = h->st;                                 // a subset call: a view of n rows
    if (ids) v.n_streams = n;
    if (mask & 3) plan_enc_analysis(plan, v, pcm, pcm_stride, nbytes, mask & 3, ids);
    if (mask & 60) plan_enc_quant(plan, v, frames_out, nbytes, frame_stride, mask >> 2, ids);
    return h->graph_mode ? plan_launch_graph(h->graphs, plan, stream) : plan_launch_direct(plan, stream);
}

// Validates the id list on the host and copies it into the workspace's id area (one cudaMemcpyAsync).  Returns an
// LC3B_* code; nothing is enqueued unless it is LC3B_OK.
static int stage_ids(lc3b_encoder* h, const int32_t* stream_ids, int n, cudaStream_t stream) {
    const EncoderState& st = h->st;
    if (!stream_ids || n < 0 || n > st.n_streams) return LC3B_ERR_INVALID_ARG;
    if (!h->id_list.take(stream_ids, n, st.n_streams)) return LC3B_ERR_INVALID_ARG;   // lc3_encoder.rs:175 (channel_index)
    if (n > 0) CU(cudaMemcpyAsync(st.ids, h->id_list.ids.data(), sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice, stream));
    return LC3B_OK;
}

extern bool lc3b_make_config(int sf, int fd, lc3b_config* c);

extern "C" {

int lc3b_encoder_workspace_bytes(int n_streams, int frame_duration, int sampling_frequency, int max_nbytes, size_t* device_bytes) {
    lc3b_config c;
    if (!device_bytes || n_streams <= 0 || max_nbytes <= 0 || max_nbytes > MAX_NBYTES ||
        lc3b_config_new(sampling_frequency, frame_duration, &c) != LC3B_OK)
        return LC3B_ERR_INVALID_ARG;
    // Lc3Encoder::new panics for 8 kHz (BandwidthDetector::new, bandwidth_detector.rs:42-56)
    if (c.fs_ind == 0) return LC3B_ERR_INVALID_ARG;
    *device_bytes = make_enc_layout(c, n_streams, max_nbytes).total;
    return LC3B_OK;
}

int lc3b_encoder_init(lc3b_encoder** out, int n_streams, int frame_duration, int sampling_frequency, int max_nbytes,
                      int device, void* dev_workspace, size_t workspace_bytes, void* cuda_stream) {
    lc3b_config c;
    if (!out || !dev_workspace || n_streams <= 0 || max_nbytes <= 0 || max_nbytes > MAX_NBYTES ||
        lc3b_config_new(sampling_frequency, frame_duration, &c) != LC3B_OK || c.fs_ind == 0)
        return LC3B_ERR_INVALID_ARG;
    const EncLayout L = make_enc_layout(c, n_streams, max_nbytes);
    if (workspace_bytes < L.total || ((uintptr_t)dev_workspace & 255) != 0) return LC3B_ERR_WORKSPACE;
    DeviceGuard guard;                        // the caller's current device is restored on return
    CU(cudaSetDevice(device));
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    uint8_t* base = (uint8_t*)dev_workspace;
    lc3b_encoder* h = new (std::nothrow) lc3b_encoder();
    if (!h) return LC3B_ERR_INVALID_ARG;
    EncoderState& st = h->st;
    st.cfg = c;
    st.n_streams = n_streams;
    st.max_nbytes = max_nbytes;
    st.device = device;
    st.ecfg = (EncConfig*)(base + L.ecfg);
    st.win = (float*)(base + L.win);
    st.dtw = (float2*)(base + L.dtw);
    st.ftw = (float2*)(base + L.ftw);
    st.perm = (int32_t*)(base + L.perm);
    st.thist = (int16_t*)(base + L.thist);
    st.xs_hist = (int16_t*)(base + L.xs_hist);
    st.x12 = (float*)(base + L.x12);
    st.x6 = (float*)(base + L.x6);
    st.estate = (int32_t*)(base + L.estate);
    st.xf = (float*)(base + L.xf);
    st.e_b = (float*)(base + L.e_b);
    st.ehand = (int32_t*)(base + L.ehand);
    st.xq = (int16_t*)(base + L.xq);
    st.qhand = (int32_t*)(base + L.qhand);
    st.lsbs = base + L.lsbs;
    st.bs_scratch = (uint32_t*)(base + L.bs_scratch);
    st.bs_words = enc_bitstream_scratch_words(c.ne, max_nbytes);
    st.stage_in = (int16_t*)(base + L.stage_in);
    st.stage_out = base + L.stage_out;
    st.ids = (int32_t*)(base + L.ids);

    const int N = c.nf / 2;
    EncConfig* hc = (EncConfig*)malloc(sizeof(EncConfig));
    float2* hd = (float2*)malloc(sizeof(float2) * N);
    float2* hf = (float2*)malloc(sizeof(float2) * N);
    int32_t* hp = (int32_t*)malloc(sizeof(int32_t) * N);
    fill_enc_config(c, hc, hd, hf, hp);
    cudaError_t e = cudaMemsetAsync(dev_workspace, 0, L.total, stream);   // the reference is handed zeroed buffers
    if (e == cudaSuccess) e = cudaMemcpyAsync(st.ecfg, hc, sizeof(EncConfig), cudaMemcpyHostToDevice, stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(st.dtw, hd, sizeof(float2) * N, cudaMemcpyHostToDevice, stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(st.ftw, hf, sizeof(float2) * N, cudaMemcpyHostToDevice, stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(st.perm, hp, sizeof(int32_t) * N, cudaMemcpyHostToDevice, stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
    free(hc); free(hd); free(hf); free(hp);
    if (e == cudaSuccess) e = prepare_enc_analysis(st);
    if (e == cudaSuccess) e = prepare_enc_quant(st);
    if (e == cudaSuccess) {
        enc_init_band_kernel<<<1, 128, 0, stream>>>(st.ecfg);
        enc_init_tables_kernel<<<1, 256, 0, stream>>>(st.ecfg, st.win);
        e = cudaGetLastError();
        if (e == cudaSuccess) e = launch_enc_init_streams(st, nullptr, n_streams, stream);
    }
    if (e != cudaSuccess) {
        delete h;
        return cuda_fail(e);
    }
    h->graph_mode = default_graph_mode(n_streams);
    *out = h;
    return LC3B_OK;
}

int lc3b_encoder_set_stage_mask(lc3b_encoder* h, int mask) {
    if (!h || mask < 1 || mask > 63) return LC3B_ERR_INVALID_ARG;
    h->stage_mask = mask;
    return LC3B_OK;
}

int lc3b_encode_frames(lc3b_encoder* h, const int16_t* pcm_in, size_t pcm_stride, uint8_t* frames_out, int nbytes,
                       size_t frame_stride, void* cuda_stream) {
    if (!h || !pcm_in || !frames_out) return LC3B_ERR_INVALID_ARG;
    const EncoderState& st = h->st;
    // the reference asserts samples_in.len() == nf (modified_dct.rs:109); a frame too small for its side information
    // underflows calc_bit_budget (spectral_quantization.rs:133) - both are panics there, invalid arguments here
    if (nbytes < 20 || nbytes > st.max_nbytes || (size_t)nbytes > frame_stride || pcm_stride < (size_t)st.cfg.nf)
        return LC3B_ERR_INVALID_ARG;
    CU(run_encode(h, pcm_in, pcm_stride, frames_out, nbytes, frame_stride, h->stage_mask, (cudaStream_t)cuda_stream));
    return LC3B_OK;
}

int lc3b_encode_frames_subset(lc3b_encoder* h, const int32_t* stream_ids, int n_rows, const int16_t* pcm_in, size_t pcm_stride,
                              uint8_t* frames_out, int nbytes, size_t frame_stride, void* cuda_stream) {
    if (!h || !stream_ids || (n_rows > 0 && (!pcm_in || !frames_out))) return LC3B_ERR_INVALID_ARG;
    const EncoderState& st = h->st;
    if (nbytes < 20 || nbytes > st.max_nbytes || (size_t)nbytes > frame_stride || pcm_stride < (size_t)st.cfg.nf)
        return LC3B_ERR_INVALID_ARG;
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    const int r = stage_ids(h, stream_ids, n_rows, stream);
    if (r != LC3B_OK || n_rows == 0) return r;
    CU(run_encode(h, pcm_in, pcm_stride, frames_out, nbytes, frame_stride, h->stage_mask, stream, st.ids, n_rows));
    return LC3B_OK;
}

int lc3b_encoder_reset_streams(lc3b_encoder* h, const int32_t* stream_ids, int n, void* cuda_stream) {
    if (!h) return LC3B_ERR_INVALID_ARG;
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    const int r = stage_ids(h, stream_ids, n, stream);
    if (r != LC3B_OK || n == 0) return r;
    CU(launch_enc_init_streams(h->st, h->st.ids, n, stream));
    return LC3B_OK;
}

int lc3b_encoder_multi_scratch_bytes(const lc3b_encoder* h, int n_frames, size_t* device_bytes) {
    if (!h || !device_bytes || n_frames < 1 || (size_t)h->st.n_streams * (size_t)n_frames > (size_t)INT32_MAX)
        return LC3B_ERR_INVALID_ARG;
    *device_bytes = enc_multi_scratch_bytes(h->st, h->st.n_streams, (long long)h->st.n_streams * n_frames);
    return LC3B_OK;
}

int lc3b_encode_stream_frames(lc3b_encoder* h, const int16_t* pcm_in, int n_frames, uint8_t* frames_out, int nbytes,
                              size_t frame_stride, void* scratch, size_t scratch_bytes, void* cuda_stream) {
    if (!h || !pcm_in || !frames_out || !scratch) return LC3B_ERR_INVALID_ARG;
    const EncoderState& st = h->st;
    if (nbytes < 20 || nbytes > st.max_nbytes || (size_t)nbytes > frame_stride || n_frames < 1 ||
        (size_t)st.n_streams * (size_t)n_frames > (size_t)INT32_MAX)
        return LC3B_ERR_INVALID_ARG;
    const long long total = (long long)st.n_streams * n_frames;
    if (scratch_bytes < enc_multi_scratch_bytes(st, st.n_streams, total) || ((uintptr_t)scratch & 255) != 0) return LC3B_ERR_WORKSPACE;
    LaunchPlan plan;                                      // the whole call is one plan: one graph launch in graph mode
    plan_enc_multi(plan, st, pcm_in, st.n_streams, st.n_streams, total, n_frames, frames_out, nbytes, frame_stride, scratch);
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    CU(h->graph_mode ? plan_launch_graph(h->graphs, plan, stream) : plan_launch_direct(plan, stream));
    return LC3B_OK;
}

int lc3b_encoder_multi_subset_scratch_bytes(const lc3b_encoder* h, int n_rows, long long total_frames, size_t* device_bytes) {
    if (!h || !device_bytes || n_rows < 0 || n_rows > h->st.n_streams || total_frames < 0 || total_frames > (long long)INT32_MAX)
        return LC3B_ERR_INVALID_ARG;
    *device_bytes = enc_multi_scratch_bytes(h->st, n_rows, total_frames);
    return LC3B_OK;
}

int lc3b_encode_stream_frames_subset(lc3b_encoder* h, const int32_t* stream_ids, const int32_t* frame_counts, int n_rows,
                                     const int16_t* pcm_in, uint8_t* frames_out, int nbytes, size_t frame_stride, void* scratch,
                                     size_t scratch_bytes, void* cuda_stream) {
    if (!h || !stream_ids || !frame_counts) return LC3B_ERR_INVALID_ARG;
    const EncoderState& st = h->st;
    if (nbytes < 20 || nbytes > st.max_nbytes || (size_t)nbytes > frame_stride) return LC3B_ERR_INVALID_ARG;
    RowTable& rt = h->row_table;
    if (!rt.take(h->id_list, stream_ids, frame_counts, n_rows, st.n_streams, (long long)INT32_MAX)) return LC3B_ERR_INVALID_ARG;
    if (rt.total == 0) return LC3B_OK;
    if (!pcm_in || !frames_out || !scratch) return LC3B_ERR_INVALID_ARG;
    if (scratch_bytes < enc_multi_scratch_bytes(st, n_rows, rt.total) || ((uintptr_t)scratch & 255) != 0) return LC3B_ERR_WORKSPACE;
    LaunchPlan plan;                                      // the whole call is one plan: one graph launch in graph mode
    plan_enc_multi(plan, st, pcm_in, n_rows, rt.n_live, rt.total, 0, frames_out, nbytes, frame_stride, scratch);
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    CU(rt.send(scratch, stream));
    CU(h->graph_mode ? plan_launch_graph(h->graphs, plan, stream) : plan_launch_direct(plan, stream));
    return LC3B_OK;
}

int lc3b_encode_frames_host(lc3b_encoder* h, const int16_t* pcm_in, size_t pcm_stride, uint8_t* frames_out, int nbytes,
                            size_t frame_stride, void* cuda_stream) {
    if (!h || !pcm_in || !frames_out) return LC3B_ERR_INVALID_ARG;
    const EncoderState& st = h->st;
    if (nbytes < 20 || nbytes > st.max_nbytes || (size_t)nbytes > frame_stride || pcm_stride < (size_t)st.cfg.nf)
        return LC3B_ERR_INVALID_ARG;
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    const size_t ns = (size_t)st.n_streams, nf = (size_t)st.cfg.nf;
    int16_t* stage = st.stage_in + (h->pipelined ? (size_t)h->buf * ns * nf : 0);
    cudaStream_t in_stream = stream;
    if (h->pipelined) {
        in_stream = h->copy_stream;
        // the staging buffer is free again once the two analysis kernels of the call that used it have run
        if (h->consumed_valid[h->buf]) CU(cudaStreamWaitEvent(in_stream, h->consumed[h->buf], 0));
    }
    if (pcm_stride == nf) CU(cudaMemcpyAsync(stage, pcm_in, ns * nf * sizeof(int16_t), cudaMemcpyHostToDevice, in_stream));
    else CU(cudaMemcpy2DAsync(stage, nf * sizeof(int16_t), pcm_in, pcm_stride * sizeof(int16_t), nf * sizeof(int16_t), ns,
                              cudaMemcpyHostToDevice, in_stream));
    if (h->pipelined) {
        CU(cudaEventRecord(h->h2d_done[h->buf], in_stream));
        CU(cudaStreamWaitEvent(stream, h->h2d_done[h->buf], 0));
    }
    // one plan for the whole call; the staging buffer counts as consumed when the call's kernels have run
    CU(run_encode(h, stage, nf, st.stage_out, nbytes, (size_t)nbytes, 63, stream));
    if (h->pipelined) {
        CU(cudaEventRecord(h->consumed[h->buf], stream));
        h->consumed_valid[h->buf] = true;
        h->buf ^= 1;
    }
    if (frame_stride == (size_t)nbytes) CU(cudaMemcpyAsync(frames_out, st.stage_out, ns * (size_t)nbytes, cudaMemcpyDeviceToHost, stream));
    else CU(cudaMemcpy2DAsync(frames_out, frame_stride, st.stage_out, (size_t)nbytes, (size_t)nbytes, ns, cudaMemcpyDeviceToHost, stream));
    return LC3B_OK;
}

// Test hook: copy out the analysis kernel's results of the last encode (device pointers, any may be NULL):
// xf [S][ne] f32 is the spectrum AFTER SNS/TNS (the quantiser's input), e_b [S][64], hand [S][8] i32, xq [S][ne] i16.
int lc3b_encoder_debug_read(lc3b_encoder* h, float* xf, float* e_b, int32_t* hand, int16_t* xq, void* cuda_stream) {
    if (!h) return LC3B_ERR_INVALID_ARG;
    const EncoderState& st = h->st;
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    const size_t ns = (size_t)st.n_streams;
    if (xf) CU(cudaMemcpyAsync(xf, st.xf, ns * st.cfg.ne * sizeof(float), cudaMemcpyDeviceToDevice, stream));
    if (e_b) CU(cudaMemcpyAsync(e_b, st.e_b, ns * 64 * sizeof(float), cudaMemcpyDeviceToDevice, stream));
    if (hand) CU(cudaMemcpyAsync(hand, st.ehand, ns * EH_WORDS * sizeof(int32_t), cudaMemcpyDeviceToDevice, stream));
    if (xq) CU(cudaMemcpyAsync(xq, st.xq, ns * st.cfg.ne * sizeof(int16_t), cudaMemcpyDeviceToDevice, stream));
    return LC3B_OK;
}

int lc3b_encoder_set_graph_mode(lc3b_encoder* h, int mode) {
    if (!h || mode < 0 || mode > 1) return LC3B_ERR_INVALID_ARG;
    h->graph_mode = mode;
    return LC3B_OK;
}

int lc3b_encoder_set_host_pipelining(lc3b_encoder* h, int on) {
    if (!h) return LC3B_ERR_INVALID_ARG;
    if (on && !h->copy_stream) {
        DeviceGuard guard;
        CU(cudaSetDevice(h->st.device));
        CU(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
        for (int i = 0; i < 2; i++) {
            CU(cudaEventCreateWithFlags(&h->h2d_done[i], cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&h->consumed[i], cudaEventDisableTiming));
        }
    }
    h->pipelined = on ? 1 : 0;
    return LC3B_OK;
}

void lc3b_encoder_destroy(lc3b_encoder* h) {
    if (!h) return;
    if (h->copy_stream) {
        cudaStreamSynchronize(h->copy_stream);
        for (int i = 0; i < 2; i++) { cudaEventDestroy(h->h2d_done[i]); cudaEventDestroy(h->consumed[i]); }
        cudaStreamDestroy(h->copy_stream);
    }
    delete h;
}

}  // extern "C"
