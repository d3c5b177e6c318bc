// lc3b engine: C ABI (include/lc3b.h) - configuration, workspace carving, launch sequencing.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <new>

#include "lc3b_common.cuh"
#include "lc3b_handles.cuh"
#include "lc3b_math.cuh"
#include "lc3_tables.h"

namespace lc3b {

static thread_local int g_last_cuda_error = 0;
int cuda_fail(cudaError_t e) {
    g_last_cuda_error = (int)e;
    return LC3B_ERR_CUDA;
}
#define CU(x) LC3B_CU(x)

int default_graph_mode(int n_streams) {
    const char* env = getenv("LC3B_GRAPH");
    if (env && (env[0] == '0' || env[0] == '1')) return env[0] - '0';
    return n_streams <= 131072 ? 1 : 0;
}

// common/config.rs:42-100
static bool make_config(int sf, int fd, lc3b_config* c) {
    static const int FS_IND[6] = {0, 1, 2, 3, 4, 4};
    static const int FS[6] = {8000, 16000, 24000, 32000, 44100, 48000};
    static const int NF75[6] = {60, 120, 180, 240, 360, 360};
    static const int NF10[6] = {80, 160, 240, 320, 480, 480};
    if (sf < 0 || sf > 5 || fd < 0 || fd > 1) return false;
    c->fs_ind = FS_IND[sf];
    c->fs = FS[sf];
    c->n_ms = fd;
    if (fd == LC3B_7P5MS) {
        c->nf = NF75[sf];
        c->ne = c->nf == 360 ? 300 : c->nf;
        c->nb = sf == LC3B_HZ8000 ? 60 : 64;
        c->z = 7 * c->nf / 30;
    } else {
        c->nf = NF10[sf];
        c->ne = c->nf == 480 ? 400 : c->nf;
        c->nb = 64;
        c->z = 3 * c->nf / 8;
    }
    return true;
}

// The LC3 tables are device-qualified in this build, so the per-config float tables that depend on them
// (window, band edges, LTPF coefficient products) are produced by a tiny init kernel (init_tables_kernel).
struct Carve {
    size_t off = 0;
    size_t take(size_t bytes) {
        size_t o = off;
        off += (bytes + 255) & ~(size_t)255;
        return o;
    }
};

struct Layout {
    size_t dcfg, win, dtw, ftw, sym_lut, spec, xq, handoff, gband, tns_list, nsym_prev, ola, ltpf_y, ltpf_xtail, ltpf_x, side, sstate, stage_in, stage_out, stage_len,
        stage_status, ids, total;
};

static Layout make_layout(const lc3b_config& c, int n_streams, int max_nbytes, bool staging = true) {
    Carve cv;
    Layout L;
    const size_t ns = (size_t)n_streams, nblk = (ns + 31) / 32;
    const int blocks = c.n_ms == LC3B_10MS ? 2 : 3;
    L.dcfg = cv.take(sizeof(DevConfig));
    L.win = cv.take(sizeof(float) * 2 * c.nf);
    L.dtw = cv.take(sizeof(float2) * (c.nf / 2));
    L.ftw = cv.take(sizeof(float2) * (c.nf / 2));
    L.sym_lut = cv.take(64 * 32);
    L.spec = cv.take(sizeof(float) * 2 * ns * c.ne);
    L.xq = cv.take(sizeof(int32_t) * nblk * c.ne * 32);
    L.handoff = cv.take(sizeof(int32_t) * ((ns + 127) / 128) * 128 * HO_WORDS);   // every thread slot of whole entropy CTAs
    L.gband = cv.take(sizeof(float) * ((ns + 127) / 128) * 128 * 64);
    L.tns_list = cv.take(sizeof(int32_t) * (2 + ((ns + 127) / 128) * 128));
    L.nsym_prev = cv.take(sizeof(int32_t) * ns);
    L.ola = cv.take(sizeof(float) * ns * (c.nf - c.z));
    L.ltpf_y = cv.take(sizeof(float) * ns * blocks * c.nf);
    L.ltpf_xtail = cv.take(sizeof(float) * ns * XTAIL_FLOATS);
    L.ltpf_x = cv.take(sizeof(float) * ns * c.nf);
    L.side = cv.take(sizeof(int32_t) * ns * SIDE_WORDS);
    L.sstate = cv.take(sizeof(int32_t) * ns * SS_WORDS);
    // staging for the host-buffer entry point (a mixed-rate handle stages for all of its buckets at once instead)
    L.stage_in = cv.take(staging ? ns * (size_t)max_nbytes : 0);
    L.stage_out = cv.take(staging ? sizeof(int16_t) * ns * c.nf * 2 : 0);   // double-buffered for the pipelined host path
    L.stage_len = cv.take(staging ? sizeof(int32_t) * ns : 0);
    L.stage_status = cv.take(staging ? sizeof(int32_t) * ns : 0);
    L.ids = cv.take(staging ? sizeof(int32_t) * ns : 0);                 // id list of a subset call (lc3b_decode_frames_subset)
    L.total = cv.off;
    return L;
}

// ---------------------------------------------------------------- device-side table construction
// Runs once per handle.  Twiddles are computed in f64 and narrowed, like the reference
// (dct_iv.rs:30-35, kissfft.rs:19-29); the window is folded with the 1/sqrt(2 nf) gain.
__global__ void init_tables_kernel(DevConfig* cfg, float* win, float2* dtw, float2* ftw) {
    const int nf = cfg->nf, N = nf / 2;
    const float* w;
    if (cfg->n_ms == LC3B_7P5MS) {
        w = nf == 60 ? LC3T_W_N60_7P5MS : nf == 120 ? LC3T_W_N120_7P5MS : nf == 180 ? LC3T_W_N180_7P5MS
            : nf == 240 ? LC3T_W_N240_7P5MS : LC3T_W_N360_7P5MS;
    } else {
        w = nf == 80 ? LC3T_W_N80_10MS : nf == 160 ? LC3T_W_N160_10MS : nf == 240 ? LC3T_W_N240_10MS
            : nf == 320 ? LC3T_W_N320_10MS : LC3T_W_N480_10MS;
    }
    const float gain = 1.0f / sqrtf(2.0f * (float)nf);
    for (int m = threadIdx.x; m < 2 * nf; m += blockDim.x) win[m] = gain * w[2 * nf - 1 - m];
    for (int i = threadIdx.x; i < N; i += blockDim.x) {
        const double t = -M_PI * (double)(8 * i + 1) / (8.0 * (double)N * 2.0);
        dtw[i] = make_float2((float)cos(t), (float)sin(t));
        const double ph = -2.0 * M_PI * (double)i / (double)N;
        ftw[i] = make_float2((float)cos(ph), (float)sin(ph));
    }
    if (threadIdx.x == 0) {
        const uint16_t* bi;
        if (cfg->n_ms == LC3B_7P5MS) {
            bi = cfg->fs_ind == 0 ? LC3T_I_8000_7P5MS : cfg->fs_ind == 1 ? LC3T_I_16000_7P5MS
                 : cfg->fs_ind == 2 ? LC3T_I_24000_7P5MS : cfg->fs_ind == 3 ? LC3T_I_32000_7P5MS : LC3T_I_48000_7P5MS;
        } else {
            bi = cfg->fs_ind == 0 ? LC3T_I_8000_10MS : cfg->fs_ind == 1 ? LC3T_I_16000_10MS
                 : cfg->fs_ind == 2 ? LC3T_I_24000_10MS : cfg->fs_ind == 3 ? LC3T_I_32000_10MS : LC3T_I_48000_10MS;
        }
        for (int b = 0; b <= cfg->nb; b++) cfg->band_idx[b] = bi[b];
        for (int b = cfg->nb + 1; b < 65; b++) cfg->band_idx[b] = cfg->ne;
        // LTPF coefficient products (long_term_post_filter.rs:204-240), 44.1 kHz uses the 48 kHz tables truncated
        static const float GAINS[4] = {0.4f, 0.35f, 0.3f, 0.25f};
        for (int g = 0; g < 4; g++) {
            for (int k = 0; k < 12; k++) cfg->ltpf_num[g][k] = 0.0f;
            for (int fr = 0; fr < 4; fr++) for (int k = 0; k < 16; k++) cfg->ltpf_den[g][fr][k] = 0.0f;
            for (int k = 0; k <= cfg->ltpf_l_num; k++) {
                float tab;
                switch (cfg->fs) {
                    case 8000: tab = LC3T_TAB_LTPF_NUM_8000[g][k]; break;
                    case 16000: tab = LC3T_TAB_LTPF_NUM_16000[g][k]; break;
                    case 24000: tab = LC3T_TAB_LTPF_NUM_24000[g][k]; break;
                    case 32000: tab = LC3T_TAB_LTPF_NUM_32000[g][k]; break;
                    default: tab = LC3T_TAB_LTPF_NUM_48000[g][k]; break;
                }
                cfg->ltpf_num[g][k] = xm(xm(0.85f, GAINS[g]), tab);
            }
            for (int fr = 0; fr < 4; fr++) {
                for (int k = 0; k <= cfg->ltpf_l_den; k++) {
                    float tab;
                    switch (cfg->fs) {
                        case 8000: tab = LC3T_TAB_LTPF_DEN_8000[fr][k]; break;
                        case 16000: tab = LC3T_TAB_LTPF_DEN_16000[fr][k]; break;
                        case 24000: tab = LC3T_TAB_LTPF_DEN_24000[fr][k]; break;
                        case 32000: tab = LC3T_TAB_LTPF_DEN_32000[fr][k]; break;
                        default: tab = LC3T_TAB_LTPF_DEN_48000[fr][k]; break;
                    }
                    cfg->ltpf_den[g][fr][k] = xm(GAINS[g], tab);
                }
            }
        }
    }
}

// coarse symbol table: for every (probability model, quotient / 32) the largest val with cum[val] <= 32 * bucket
// (arithmetic_codec.rs:82-85); the entropy kernel refines from there against the cumulative table in shared memory
__global__ void init_sym_lut_kernel(uint8_t* lut) {
    const int pki = blockIdx.x;
    for (int b = threadIdx.x; b < 32; b += blockDim.x) {
        int val = 16;
        while (LC3T_AC_SPEC_CUMFREQ[pki][val] > 32 * b) val--;
        lut[pki * 32 + b] = (uint8_t)val;
    }
}

// The state a stream starts from.  ids == nullptr: every stream, whose rows lc3b_decoder_init has just zeroed with the
// rest of the workspace; otherwise the n listed streams (lc3b_decoder_reset_streams), whose persistent rows are zeroed
// here first - one warp per stream.
__global__ void init_streams_kernel(DecoderState st, const int32_t* ids, int n) {
    const int lane = threadIdx.x & 31;
    const int i = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    if (i >= n) return;
    const int s = ids ? ids[i] : i;
    const size_t S = (size_t)st.n_streams;
    if (ids) {
        const int ne = st.cfg.ne, nf = st.cfg.nf;
        const int hist = (st.cfg.n_ms == LC3B_10MS ? 2 : 3) * nf;
        for (int k = lane; k < ne; k += 32) { st.spec[(size_t)s * ne + k] = 0.0f; st.spec[(S + s) * ne + k] = 0.0f; }
        for (int k = lane; k < nf - st.cfg.z; k += 32) st.ola[(size_t)s * (nf - st.cfg.z) + k] = 0.0f;
        for (int k = lane; k < hist; k += 32) st.ltpf_y[(size_t)s * hist + k] = 0.0f;
        for (int k = lane; k < XTAIL_FLOATS; k += 32) st.ltpf_xtail[(size_t)s * XTAIL_FLOATS + k] = 0.0f;
        for (int k = lane; k < nf; k += 32) st.ltpf_x[(size_t)s * nf + k] = 0.0f;
        if (lane < SIDE_WORDS) st.side[(size_t)s * SIDE_WORDS + lane] = 0;
        if (lane == 0) st.nsym_prev[s] = 0;
    }
    if (lane != 0) return;
    int32_t* ss = st.sstate + (size_t)s * SS_WORDS;
    ss[SS_SLOT] = 0;
    ss[SS_PLC_LOST] = 0;
    ss[SS_PLC_ALPHA] = (int32_t)f2u(1.0f);     // packet_loss_concealment.rs:31-33
    ss[SS_PLC_SEED] = 24607;
    ss[SS_LTPF_PREV] = 4 << 8;
    ss[SS_LTPF_PINT] = 0;
    ss[SS_LTPF_PFR] = 0;
    ss[SS_LTPF_BLK] = 0;
}

static cudaError_t launch_init_streams(const DecoderState& st, const int32_t* ids, int n, cudaStream_t stream) {
    init_streams_kernel<<<(unsigned)((n + 7) / 8), 256, 0, stream>>>(st, ids, n);
    return cudaGetLastError();
}

static void fill_host_config(const lc3b_config& c, DevConfig* d) {
    memset(d, 0, sizeof(*d));
    d->fs_ind = c.fs_ind; d->fs = c.fs; d->ne = c.ne; d->nb = c.nb; d->nf = c.nf; d->z = c.z; d->n_ms = c.n_ms;
    static const int NBITS_BW[5] = {0, 1, 2, 2, 3};           // side_info_reader.rs:11
    d->nbits_bw = NBITS_BW[c.fs_ind];
    int lg = 0;
    while ((1 << lg) < c.ne / 2) lg++;                        // ((ne/2) as f32).log2().ceil(), side_info_reader.rs:50
    d->lastnz_bits = lg;
    d->n_fft = c.nf / 2;
    // Stockham stage radices: 4s, then 2, 3s, 5s
    int n = d->n_fft, i = 0;
    while (n % 4 == 0) { d->fft_radix[i++] = 4; n /= 4; }
    while (n % 2 == 0) { d->fft_radix[i++] = 2; n /= 2; }
    while (n % 3 == 0) { d->fft_radix[i++] = 3; n /= 3; }
    while (n % 5 == 0) { d->fft_radix[i++] = 5; n /= 5; }
    switch (c.fs) {                                            // long_term_post_filter.rs:104-134
        case 8000: case 16000: d->ltpf_l_den = 4; break;
        case 24000: d->ltpf_l_den = 6; break;
        case 32000: d->ltpf_l_den = 8; break;
        case 44100: d->ltpf_l_den = 11; break;
        default: d->ltpf_l_den = 12; break;
    }
    d->ltpf_l_num = d->ltpf_l_den - 2;
    if (c.n_ms == LC3B_10MS) { d->ltpf_blocks = 2; d->ltpf_norm = c.nf / 4; } else { d->ltpf_blocks = 3; d->ltpf_norm = c.nf / 3; }
    d->ltpf_s2p5 = c.fs == 44100 ? 48000 / 400 : c.fs / 400;
    for (int k = 0; k < 400; k++) d->gg_table[k] = powf_msun(10.0f, xd((float)(k - 245), 28.0f));   // global_gain.rs:19-20
    {                                                          // noise_filling.rs:49 composed n times
        uint32_t a = 1, cc = 0;
        d->nf_lcg[0] = (1u << 16);
        for (int n = 1; n <= MAX_NE; n++) {
            a = (a * 31821u) & 0xffffu;
            cc = (cc * 31821u + 13849u) & 0xffffu;
            d->nf_lcg[n] = (a << 16) | cc;
        }
    }
    const float step = (float)(M_PI / 17.0);                   // temporal_noise_shaping.rs:38-45
    for (int k = 0; k < 17; k++) d->tns_sin[k] = (float)sin((double)xm(step, (float)(k - 8)));
}

__host__ __device__ inline float math_dispatch(int which, float x, float y) {
    switch (which) {
        case 0: return powf_msun(x, y);
        case 1: return log2f_msun(x);
        case 2: return log10f_msun(x);
        case 3: return exp2f_msun(x);
        case 4: return asinf_msun(x);
        case 5: return exp2_raw_fm(x);
        default: return powi_nt(x, (int32_t)y);
    }
}
__global__ void math_kernel(int which, const float* x, const float* y, float* out, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = math_dispatch(which, x[i], y ? y[i] : 0.0f);
}

}  // namespace lc3b

using namespace lc3b;


extern "C" {

const char* lc3b_version(void) { return "lc3b 0.1 (sm_100a)"; }
int lc3b_last_cuda_error(void) { return g_last_cuda_error; }

int lc3b_config_new(int sampling_frequency, int frame_duration, lc3b_config* out) {
    if (!out || !make_config(sampling_frequency, frame_duration, out)) return LC3B_ERR_INVALID_ARG;
    return LC3B_OK;
}

int lc3b_decoder_workspace_bytes(int n_streams, int frame_duration, int sampling_frequency, int max_nbytes,
                                 size_t* device_bytes) {
    return lc3b::decoder_workspace_bytes(n_streams, frame_duration, sampling_frequency, max_nbytes, true, device_bytes);
}

int lc3b_decoder_init(lc3b_decoder** out, int n_streams, int frame_duration, int sampling_frequency, int max_nbytes,
                      int device, void* dev_workspace, size_t workspace_bytes, void* cuda_stream) {
    return lc3b::decoder_init(out, n_streams, frame_duration, sampling_frequency, max_nbytes, device, dev_workspace,
                              workspace_bytes, cuda_stream, true);
}

}  // extern "C"

namespace lc3b {

bool config_new(int sf, int fd, lc3b_config* c) { return make_config(sf, fd, c); }

int decoder_workspace_bytes(int n_streams, int frame_duration, int sampling_frequency, int max_nbytes, bool staging,
                            size_t* device_bytes) {
    lc3b_config c;
    if (!device_bytes || n_streams <= 0 || max_nbytes <= 0 || max_nbytes > MAX_NBYTES ||
        !make_config(sampling_frequency, frame_duration, &c))
        return LC3B_ERR_INVALID_ARG;
    *device_bytes = make_layout(c, n_streams, max_nbytes, staging).total;
    return LC3B_OK;
}

int decoder_init(lc3b_decoder** out, int n_streams, int frame_duration, int sampling_frequency, int max_nbytes,
                 int device, void* dev_workspace, size_t workspace_bytes, void* cuda_stream, bool staging) {
    lc3b_config c;
    if (!out || !dev_workspace || n_streams <= 0 || max_nbytes <= 0 || max_nbytes > MAX_NBYTES ||
        !make_config(sampling_frequency, frame_duration, &c))
        return LC3B_ERR_INVALID_ARG;
    const Layout L = make_layout(c, n_streams, max_nbytes, staging);
    if (workspace_bytes < L.total || ((uintptr_t)dev_workspace & 255) != 0) return LC3B_ERR_WORKSPACE;
    DeviceGuard guard;                        // the caller's current device is restored on return
    CU(cudaSetDevice(device));
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    uint8_t* base = (uint8_t*)dev_workspace;
    lc3b_decoder* h = new (std::nothrow) lc3b_decoder();
    if (!h) return LC3B_ERR_INVALID_ARG;
    DecoderState& st = h->st;
    st.cfg = c;
    st.n_streams = n_streams;
    st.n_blocks32 = (n_streams + 31) / 32;
    st.max_nbytes = max_nbytes;
    st.device = device;
    st.dcfg = (DevConfig*)(base + L.dcfg);
    st.win = (float*)(base + L.win);
    st.dtw = (float2*)(base + L.dtw);
    st.ftw = (float2*)(base + L.ftw);
    st.sym_lut = base + L.sym_lut;
    st.spec = (float*)(base + L.spec);
    st.xq = (int32_t*)(base + L.xq);
    st.handoff = (int32_t*)(base + L.handoff);
    st.gband = (float*)(base + L.gband);
    st.tns_list = (int32_t*)(base + L.tns_list);
    st.nsym_prev = (int32_t*)(base + L.nsym_prev);
    st.ola = (float*)(base + L.ola);
    st.ltpf_y = (float*)(base + L.ltpf_y);
    st.ltpf_xtail = (float*)(base + L.ltpf_xtail);
    st.ltpf_x = (float*)(base + L.ltpf_x);
    st.side = (int32_t*)(base + L.side);
    st.sstate = (int32_t*)(base + L.sstate);
    st.stage_in = base + L.stage_in;
    st.stage_out = (int16_t*)(base + L.stage_out);
    st.stage_len = (int32_t*)(base + L.stage_len);
    st.stage_status = (int32_t*)(base + L.stage_status);
    st.ids = staging ? (int32_t*)(base + L.ids) : nullptr;
    st.trace = nullptr;
    st.trace_x = nullptr;
    st.fixed_slot = -1;
    st.dequant_mode = 0;
    st.synth_mode = 0;
    st.no_ltpf = 0;
    st.min_nbytes = 0;
    st.sm_count = 148;
    {
        int sms = 0;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) == cudaSuccess && sms > 0) st.sm_count = sms;
    }

    DevConfig hc;
    fill_host_config(c, &hc);
    cudaError_t e = cudaMemsetAsync(dev_workspace, 0, L.total, stream);   // the reference is handed zeroed buffers
    if (e == cudaSuccess) e = cudaMemcpyAsync(st.dcfg, &hc, sizeof(hc), cudaMemcpyHostToDevice, stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(stream);               // hc is a stack object
    if (e == cudaSuccess) e = prepare_entropy(st);
    if (e == cudaSuccess) e = prepare_synth(st);
    if (e == cudaSuccess) e = prepare_multi(st);
    if (e == cudaSuccess) {
        init_tables_kernel<<<1, 256, 0, stream>>>(st.dcfg, st.win, st.dtw, st.ftw);
        init_sym_lut_kernel<<<64, 32, 0, stream>>>(st.sym_lut);
        e = cudaGetLastError();
        if (e == cudaSuccess) e = launch_init_streams(st, nullptr, n_streams, stream);
    }
    if (e != cudaSuccess) {
        delete h;
        return cuda_fail(e);
    }
    h->graph_mode = default_graph_mode(n_streams);
    *out = h;
    return LC3B_OK;
}

}  // namespace lc3b

extern "C" {

int lc3b_decoder_set_host_pipelining(lc3b_decoder* h, int on) {
    if (!h) return LC3B_ERR_INVALID_ARG;
    if (!on && h->pipelined) {
        // copies still in flight read the staging halves the next (unpipelined) call writes: let them land first
        for (int i = 0; i < 2; i++)
            if (h->d2h_pending[i]) { CU(cudaEventSynchronize(h->d2h_done[i])); h->d2h_pending[i] = false; }
    }
    if (on && !h->copy_stream) {
        DeviceGuard guard;
        CU(cudaSetDevice(h->st.device));
        CU(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
        for (int i = 0; i < 2; i++) {
            CU(cudaEventCreateWithFlags(&h->compute_done[i], cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&h->d2h_done[i], cudaEventDisableTiming));
        }
    }
    h->pipelined = on ? 1 : 0;
    return LC3B_OK;
}

int lc3b_decoder_host_fence(lc3b_decoder* h, void* cuda_stream) {
    if (!h) return LC3B_ERR_INVALID_ARG;
    // d2h_pending stays set: a later decode on ANOTHER stream than the one fenced here must still wait for the
    // staging half it overwrites (waiting twice on a completed event costs nothing)
    for (int i = 0; i < 2; i++)
        if (h->d2h_pending[i]) CU(cudaStreamWaitEvent((cudaStream_t)cuda_stream, h->d2h_done[i], 0));
    return LC3B_OK;
}

int lc3b_decoder_set_graph_mode(lc3b_decoder* h, int mode) {
    if (!h || mode < 0 || mode > 1) return LC3B_ERR_INVALID_ARG;
    h->graph_mode = mode;
    return LC3B_OK;
}

int lc3b_decoder_set_split(lc3b_decoder* h, int k) {
    if (!h || !(k == 0 || k == 1 || k == 2 || k == 4)) return LC3B_ERR_INVALID_ARG;
    h->split = k;
    return LC3B_OK;
}

// long_term_post_filter.rs:142-161: the filter's gain is the table row (0.0, 0) once the (10 ms-equivalent) frame bits reach
// 560 + 80 * fs_ind - from there on is_active can be set in the bitstream but the filter passes its input through
static bool ltpf_impossible(const lc3b_config& c, int nbytes) {
    const int nbits = nbytes * 8;
    const int t_nbits = c.n_ms == LC3B_7P5MS ? (int)round((double)nbits * 10.0 / 7.5) : nbits;
    return t_nbits >= 560 + c.fs_ind * 80;
}

int lc3b_decoder_set_min_nbytes(lc3b_decoder* h, int min_nbytes) {
    if (!h || min_nbytes < 0 || min_nbytes > h->st.max_nbytes) return LC3B_ERR_INVALID_ARG;
    h->st.min_nbytes = min_nbytes;
    h->st.no_ltpf = (min_nbytes > 0 && ltpf_impossible(h->st.cfg, min_nbytes)) ? 1 : 0;
    return LC3B_OK;
}

int lc3b_decoder_set_synth_mode(lc3b_decoder* h, int mode) {
    if (!h || mode < 0 || mode > 1) return LC3B_ERR_INVALID_ARG;
    h->st.synth_mode = mode;
    return LC3B_OK;
}

int lc3b_decoder_set_dequant_mode(lc3b_decoder* h, int mode) {
    if (!h || mode < 0 || mode > 2) return LC3B_ERR_INVALID_ARG;
    h->st.dequant_mode = mode;
    return LC3B_OK;
}

int lc3b_decoder_graph_stats(const lc3b_decoder* h, uint64_t* hits, uint64_t* updates, uint64_t* builds) {
    if (!h) return LC3B_ERR_INVALID_ARG;
    if (hits) *hits = h->graphs.hits;
    if (updates) *updates = h->graphs.updates;
    if (builds) *builds = h->graphs.builds;
    return LC3B_OK;
}

int lc3b_decoder_set_stage_mask(lc3b_decoder* h, int mask) {
    if (!h || mask < 1 || mask > 7) return LC3B_ERR_INVALID_ARG;
    h->stage_mask = mask;
    return LC3B_OK;
}

int lc3b_decoder_multi_scratch_bytes(const lc3b_decoder* h, int n_frames, size_t* device_bytes) {
    if (!h || !device_bytes || n_frames <= 0) return LC3B_ERR_INVALID_ARG;
    if ((long long)h->st.n_streams * n_frames > 0x7fffffffLL / 512) return LC3B_ERR_INVALID_ARG;   // 32-bit unit indices
    *device_bytes = multi_scratch_bytes(h->st, h->st.n_streams, (long long)h->st.n_streams * n_frames);
    return LC3B_OK;
}

int lc3b_decode_stream_frames(lc3b_decoder* h, int bits_per_sample, const uint8_t* frames, const int32_t* frame_nbytes,
                              int nbytes, size_t frame_stride, int n_frames, int16_t* pcm_out, int32_t* status_out,
                              void* scratch, size_t scratch_bytes, void* cuda_stream) {
    if (!h || !frames || !pcm_out || !scratch) return LC3B_ERR_INVALID_ARG;
    if (bits_per_sample != 16) return LC3B_ERR_BITS_PER_SAMPLE;             // lc3_decoder.rs:80
    const DecoderState& st = h->st;
    if (n_frames <= 0 || nbytes <= 0 || nbytes > st.max_nbytes || frame_stride < (size_t)nbytes) return LC3B_ERR_INVALID_ARG;
    if ((long long)st.n_streams * n_frames > 0x7fffffffLL / 512) return LC3B_ERR_INVALID_ARG;
    const long long total = (long long)st.n_streams * n_frames;
    if (scratch_bytes < multi_scratch_bytes(st, st.n_streams, total) || ((uintptr_t)scratch & 255) != 0) return LC3B_ERR_WORKSPACE;
    CU(launch_decode_multi(st, frames, frame_nbytes, nbytes, frame_stride, st.n_streams, st.n_streams, total, n_frames, pcm_out,
                           status_out, scratch, (cudaStream_t)cuda_stream, h->split == 1 ? nullptr : &h->lanes));
    return LC3B_OK;
}

static constexpr long long MULTI_MAX_UNITS = 0x7fffffffLL / 512;          // 32-bit unit indices

int lc3b_decoder_multi_subset_scratch_bytes(const lc3b_decoder* h, int n_rows, long long total_frames, size_t* device_bytes) {
    if (!h || !device_bytes || n_rows < 0 || n_rows > h->st.n_streams || total_frames < 0 || total_frames > MULTI_MAX_UNITS)
        return LC3B_ERR_INVALID_ARG;
    *device_bytes = multi_scratch_bytes(h->st, n_rows, total_frames);
    return LC3B_OK;
}

int lc3b_decode_stream_frames_subset(lc3b_decoder* h, int bits_per_sample, const int32_t* stream_ids, const int32_t* frame_counts,
                                     int n_rows, const uint8_t* frames, const int32_t* frame_nbytes, int nbytes,
                                     size_t frame_stride, int16_t* pcm_out, int32_t* status_out, void* scratch,
                                     size_t scratch_bytes, void* cuda_stream) {
    if (!h || !stream_ids || !frame_counts) return LC3B_ERR_INVALID_ARG;
    if (bits_per_sample != 16) return LC3B_ERR_BITS_PER_SAMPLE;             // lc3_decoder.rs:80
    const DecoderState& st = h->st;
    if (nbytes <= 0 || nbytes > st.max_nbytes || frame_stride < (size_t)nbytes) return LC3B_ERR_INVALID_ARG;
    RowTable& rt = h->row_table;
    if (!rt.take(h->id_list, stream_ids, frame_counts, n_rows, st.n_streams, MULTI_MAX_UNITS)) return LC3B_ERR_INVALID_ARG;
    if (rt.total == 0) return LC3B_OK;
    if (!frames || !pcm_out || !scratch) return LC3B_ERR_INVALID_ARG;
    if (scratch_bytes < multi_scratch_bytes(st, n_rows, rt.total) || ((uintptr_t)scratch & 255) != 0) return LC3B_ERR_WORKSPACE;
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    CU(rt.send(scratch, stream));
    CU(launch_decode_multi(st, frames, frame_nbytes, nbytes, frame_stride, n_rows, rt.n_live, rt.total, 0, pcm_out, status_out,
                           scratch, stream, h->split == 1 ? nullptr : &h->lanes));
    return LC3B_OK;
}

int lc3b_decoder_set_trace(lc3b_decoder* h, int32_t* trace, int32_t* x) {
    if (!h) return LC3B_ERR_INVALID_ARG;
    h->st.trace = trace;
    h->st.trace_x = x;
    return LC3B_OK;
}

// one decode_frame per stream (ids == nullptr, n = every stream of the handle) or per row of a subset call (n rows, row u
// = stream ids[u], ids in device memory): the call's kernels as a plan, issued directly or as a cached graph
static cudaError_t run_decode(lc3b_decoder* h, const uint8_t* frames, const int32_t* frame_nbytes, int nbytes, size_t frame_stride,
                              int16_t* pcm_out, size_t pcm_stride, int32_t* status_out, int stage_mask, cudaStream_t stream,
                              const int32_t* ids = nullptr, int n = 0) {
    LaunchPlan plan;
    // Sub-batches.  The three kernels are bound by different things (integer ALU / dependent-instruction latency / the
    // memory-instruction path) and each ends in a ragged last wave of CTAs that are serial chains as long as a full
    // wave's; issued as K independent sub-batches - K chains of kernels that only meet at the end of the call - one
    // sub-batch's kernels fill the SMs the other's tail leaves idle and share them with a kernel that wants a different
    // pipe.  Measured at 262 144 streams of 48 kHz / 150 B: 1.87 ms as one batch, 1.70 ms as two, 1.69 ms as four
    // (tools/exp_split_overlap.py); 131 072 streams 1.11 -> 0.91 ms, 65 536 streams 0.57 -> 0.53 ms, no difference at 32 768 and
    // below.  Streams are independent (lc3_decoder.rs:62-69), so any split computes the same bits.
    if (!ids) n = h->st.n_streams;
    int k_sub = h->split;
    if (k_sub == 0) {
        static const int env = [] { const char* e = getenv("LC3B_SPLIT"); return e ? atoi(e) : 0; }();
        k_sub = env > 0 ? env : (n >= decode_split_min_streams() ? PLAN_MAX_LANES : 1);
    }
    if (k_sub > PLAN_MAX_LANES) k_sub = PLAN_MAX_LANES;
    if (use_dequant_warp(n, h->st.dequant_mode)) k_sub = 1;            // the small-batch kernels share one list per handle
    int part = ((n + k_sub - 1) / k_sub + 127) & ~127;                // whole entropy CTAs
    if (k_sub <= 1 || part >= n) { k_sub = 1; part = n; }
    for (int k = 0, base = 0; k < k_sub && base < n; k++, base += part) {
        int count = k_sub == 1 ? -1 : (n - base < part ? n - base : part);
        plan.lane = k;
        const int first = plan.n;
        if (ids && count < 0) count = n;                                // with an id list the launch size is the call's, not the handle's
        if (stage_mask & 3)
            plan_entropy(plan, h->st, frames, frame_nbytes, nbytes, frame_stride, status_out, stage_mask & 3, base, count, -1, ids, n);
        if (stage_mask & 4) {
            if (plan_synth(plan, h->st, pcm_out, pcm_stride, plan.n > first ? plan.n - 1 : -1, base, count, ids) < 0) return cudaErrorInvalidValue;
        }
    }
    return h->graph_mode ? plan_launch_graph(h->graphs, plan, stream) : plan_launch_direct(plan, stream, &h->lanes);
}

int lc3b_decode_frames(lc3b_decoder* h, int bits_per_sample, const uint8_t* frames, const int32_t* frame_nbytes,
                       int nbytes, size_t frame_stride, int16_t* pcm_out, size_t pcm_stride, int32_t* status_out,
                       void* cuda_stream) {
    if (!h || !frames || !pcm_out) return LC3B_ERR_INVALID_ARG;
    if (bits_per_sample != 16) return LC3B_ERR_BITS_PER_SAMPLE;                       // lc3_decoder.rs:80
    const DecoderState& st = h->st;
    if (nbytes < 0 || nbytes > st.max_nbytes || (size_t)nbytes > frame_stride || pcm_stride < (size_t)st.cfg.nf)
        return LC3B_ERR_INVALID_ARG;
    if (!frame_nbytes && nbytes < st.min_nbytes) return LC3B_ERR_INVALID_ARG;       // lc3b_decoder_set_min_nbytes
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    CU(run_decode(h, frames, frame_nbytes, nbytes, frame_stride, pcm_out, pcm_stride, status_out, h->stage_mask, stream));
    return LC3B_OK;
}

// Validates the id list on the host and copies it into the workspace's id area (one cudaMemcpyAsync).  Returns an
// LC3B_* code; nothing is enqueued unless it is LC3B_OK.
static int stage_ids(lc3b_decoder* h, const int32_t* stream_ids, int n, cudaStream_t stream) {
    const DecoderState& st = h->st;
    if (!stream_ids || n < 0 || n > st.n_streams || !st.ids) return LC3B_ERR_INVALID_ARG;
    if (!h->id_list.take(stream_ids, n, st.n_streams)) return LC3B_ERR_INVALID_ARG;   // lc3_decoder.rs:228
    if (n > 0) CU(cudaMemcpyAsync(st.ids, h->id_list.ids.data(), sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice, stream));
    return LC3B_OK;
}

int lc3b_decode_frames_subset(lc3b_decoder* h, int bits_per_sample, const int32_t* stream_ids, int n_rows, const uint8_t* frames,
                              const int32_t* frame_nbytes, int nbytes, size_t frame_stride, int16_t* pcm_out, size_t pcm_stride,
                              int32_t* status_out, void* cuda_stream) {
    if (!h || !stream_ids || (n_rows > 0 && (!frames || !pcm_out))) return LC3B_ERR_INVALID_ARG;
    if (bits_per_sample != 16) return LC3B_ERR_BITS_PER_SAMPLE;                       // lc3_decoder.rs:80
    const DecoderState& st = h->st;
    if (nbytes < 0 || nbytes > st.max_nbytes || (size_t)nbytes > frame_stride || pcm_stride < (size_t)st.cfg.nf)
        return LC3B_ERR_INVALID_ARG;
    if (!frame_nbytes && nbytes < st.min_nbytes) return LC3B_ERR_INVALID_ARG;       // lc3b_decoder_set_min_nbytes
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    const int r = stage_ids(h, stream_ids, n_rows, stream);
    if (r != LC3B_OK || n_rows == 0) return r;
    CU(run_decode(h, frames, frame_nbytes, nbytes, frame_stride, pcm_out, pcm_stride, status_out, h->stage_mask, stream, st.ids, n_rows));
    return LC3B_OK;
}

int lc3b_decoder_reset_streams(lc3b_decoder* h, const int32_t* stream_ids, int n, void* cuda_stream) {
    if (!h) return LC3B_ERR_INVALID_ARG;
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    const int r = stage_ids(h, stream_ids, n, stream);
    if (r != LC3B_OK || n == 0) return r;
    CU(launch_init_streams(h->st, h->st.ids, n, stream));
    return LC3B_OK;
}

int lc3b_decode_frames_host(lc3b_decoder* h, int bits_per_sample, const uint8_t* frames, const int32_t* frame_nbytes,
                            int nbytes, size_t frame_stride, int16_t* pcm_out, size_t pcm_stride, int32_t* status_out,
                            void* cuda_stream) {
    if (!h || !frames || !pcm_out) return LC3B_ERR_INVALID_ARG;
    if (bits_per_sample != 16) return LC3B_ERR_BITS_PER_SAMPLE;
    const DecoderState& st = h->st;
    if (nbytes < 0 || nbytes > st.max_nbytes || (size_t)nbytes > frame_stride || pcm_stride < (size_t)st.cfg.nf)
        return LC3B_ERR_INVALID_ARG;
    if (!frame_nbytes && nbytes < st.min_nbytes) return LC3B_ERR_INVALID_ARG;
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    const size_t ns = (size_t)st.n_streams;
    // frames: one strided copy packs the rows to pitch `nbytes`
    // (a pitched copy of many short rows is far slower than one linear copy, so the dense case takes the linear path)
    if (frame_stride == (size_t)nbytes) CU(cudaMemcpyAsync(st.stage_in, frames, ns * (size_t)nbytes, cudaMemcpyHostToDevice, stream));
    else CU(cudaMemcpy2DAsync(st.stage_in, (size_t)nbytes, frames, frame_stride, (size_t)nbytes, ns, cudaMemcpyHostToDevice, stream));
    if (frame_nbytes) CU(cudaMemcpyAsync(st.stage_len, frame_nbytes, sizeof(int32_t) * ns, cudaMemcpyHostToDevice, stream));
    const size_t out_elems = ns * (size_t)st.cfg.nf;
    int16_t* stage = st.stage_out + (h->pipelined ? (size_t)h->buf * out_elems : 0);
    cudaStream_t out_stream = stream;
    if (h->pipelined) {
        // the staging half about to be overwritten must have left the device (copy issued two calls ago)
        if (h->d2h_pending[h->buf]) CU(cudaStreamWaitEvent(stream, h->d2h_done[h->buf], 0));
        out_stream = h->copy_stream;
    }
    CU(run_decode(h, st.stage_in, frame_nbytes ? st.stage_len : nullptr, nbytes, (size_t)nbytes, stage, (size_t)st.cfg.nf,
                  status_out ? st.stage_status : nullptr, 7, stream));
    if (h->pipelined) {
        CU(cudaEventRecord(h->compute_done[h->buf], stream));
        CU(cudaStreamWaitEvent(out_stream, h->compute_done[h->buf], 0));
    }
    if (pcm_stride == (size_t)st.cfg.nf)
        CU(cudaMemcpyAsync(pcm_out, stage, out_elems * sizeof(int16_t), cudaMemcpyDeviceToHost, out_stream));
    else
        CU(cudaMemcpy2DAsync(pcm_out, pcm_stride * sizeof(int16_t), stage, (size_t)st.cfg.nf * sizeof(int16_t),
                             (size_t)st.cfg.nf * sizeof(int16_t), ns, cudaMemcpyDeviceToHost, out_stream));
    if (h->pipelined) {
        CU(cudaEventRecord(h->d2h_done[h->buf], out_stream));
        h->d2h_pending[h->buf] = true;
        h->buf ^= 1;
    }
    if (status_out) CU(cudaMemcpyAsync(status_out, st.stage_status, sizeof(int32_t) * ns, cudaMemcpyDeviceToHost, stream));
    return LC3B_OK;
}

int lc3b_decoder_get_spectrum(lc3b_decoder* h, float* out, void* cuda_stream) {
    if (!h || !out) return LC3B_ERR_INVALID_ARG;
    // the slot differs per stream; gather on the device
    extern void lc3b_gather_spectrum(const DecoderState&, float*, cudaStream_t);
    lc3b_gather_spectrum(h->st, out, (cudaStream_t)cuda_stream);
    CU(cudaGetLastError());
    return LC3B_OK;
}

void lc3b_decoder_destroy(lc3b_decoder* h) {
    if (!h) return;
    if (h->copy_stream) {
        cudaStreamSynchronize(h->copy_stream);
        for (int i = 0; i < 2; i++) { cudaEventDestroy(h->compute_done[i]); cudaEventDestroy(h->d2h_done[i]); }
        cudaStreamDestroy(h->copy_stream);
    }
    delete h;
}

int lc3b_selftest_math_host(int which, const float* x, const float* y, float* out, int n) {
    if (!x || !out || n < 0 || which < 0 || which > 6) return LC3B_ERR_INVALID_ARG;
    for (int i = 0; i < n; i++) out[i] = lc3b::math_dispatch(which, x[i], y ? y[i] : 0.0f);
    return LC3B_OK;
}

int lc3b_selftest_math_device(int which, const float* x, const float* y, float* out, int n, void* cuda_stream) {
    if (!x || !out || n < 0 || which < 0 || which > 6) return LC3B_ERR_INVALID_ARG;
    lc3b::math_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)cuda_stream>>>(which, x, y, out, n);
    CU(cudaGetLastError());
    return LC3B_OK;
}

}  // extern "C"

namespace lc3b {
// after any decode call (frame by frame or time-parallel) the stream's SS_SLOT names the slot of its last good spectrum,
// which is also what the last frame's IMDCT read unless that frame was concealed (then: the spectrum it was faded from)
__global__ void gather_spectrum_kernel(const float* spec, const int32_t* sstate, float* out, int n_streams, int ne) {
    const int s = blockIdx.x;
    const int slot = sstate[(size_t)s * SS_WORDS + SS_SLOT];
    const float* sp = spec + ((size_t)slot * n_streams + s) * ne;
    for (int k = threadIdx.x; k < ne; k += blockDim.x) out[(size_t)s * ne + k] = sp[k];
}
}  // namespace lc3b

void lc3b_gather_spectrum(const lc3b::DecoderState& st, float* out, cudaStream_t stream) {
    lc3b::gather_spectrum_kernel<<<st.n_streams, 128, 0, stream>>>(st.spec, st.sstate, out, st.n_streams, st.cfg.ne);
}
