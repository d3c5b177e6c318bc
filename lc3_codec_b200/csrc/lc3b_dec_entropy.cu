// lc3b engine, decoder kernels 1a and 1b: bitstream -> shaped spectrum, one THREAD per frame.
//
// Replaces, per stream, the first half of DecoderChannel::decode (src/decoder/lc3_decoder.rs:73-135):
//   side_info_reader::read            src/decoder/side_info_reader.rs:29
//   arithmetic_codec::decode          src/decoder/arithmetic_codec.rs:109 (range decoder, TNS data, spectral tuples,
//                                     residual / lsb-mode bits, noise-filling seed, zero-frame flag)
//   residual_spectrum::decode         src/decoder/residual_spectrum.rs:13
//   noise_filling::apply_noise_filling src/decoder/noise_filling.rs:18
//   global_gain::apply_global_gain    src/decoder/global_gain.rs:15
//   temporal_noise_shaping            src/decoder/temporal_noise_shaping.rs:24
//   spectral_noise_shaping::decode    src/decoder/spectral_noise_shaping.rs:21
// Everything here is a serial recurrence per frame (range state, context chain, LCG, lattice), so the
// parallel axis is frames: lane = frame, a warp = 32 consecutive streams, all lanes walk the same line
// index k so that the per-line traffic is coalesced:
//   * the frame bytes of the CTA are staged once into shared memory (rows padded to an odd word count);
//   * pass 1 (entropy) writes integers to a lane-interleaved scratch  xq[warp][k / 4][lane][k % 4]  (a tuple is one
//     8-byte store, four lines are one 16-byte load for pass 2; a warp's accesses are contiguous);
//   * pass 2 (dequantise + noise fill + gain + TNS lattice + SNS gain) streams them back and writes the f32
//     spectrum four lines at a time (16 bytes per thread) into the stream-major slot  spec[slot][stream][k].
// The spectrum slot written is the stream's INACTIVE one; it becomes the active slot (= PLC "last good",
// packet_loss_concealment.rs:50) only if the frame decoded without error, so concealment needs no copy.
// All f32 arithmetic uses contraction-proof ops in the reference's order: the spectrum is bit-exact.
#include <stdlib.h>
#include <string.h>

#include <type_traits>

#include "lc3b_common.cuh"
#include "lc3b_math.cuh"
#include "lc3b_plan.cuh"
#include "lc3_tables.h"

namespace lc3b {


// ---------------------------------------------------------------- bit reader over one staged frame (buffer_reader.rs)
struct Reader {
    const uint8_t* buf;   // shared-memory row
    int len;              // buf_in.len()
    int head;             // head_byte_cursor
    int tail;             // tail_bit_cursor
    uint64_t tw;          // window of not-yet-consumed tail bits, LSB = next bit; (tail + tw_n) % 8 == 0 always
    int tw_n;             // valid bits in tw

    __device__ __forceinline__ void refill() {                         // up to 4 more bytes, counted from the end
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const int idx = len - 1 - ((tail + tw_n) >> 3);
            const uint32_t byte = idx >= 0 ? buf[idx] : 0u;
            tw |= (uint64_t)byte << tw_n;
            tw_n += 8;
        }
    }
    __device__ __forceinline__ bool head_byte(uint32_t& out) {          // :42
        if (head >= len) return false;
        out = buf[head++];
        return true;
    }
    __device__ __forceinline__ bool tail_bool(int& bit) {               // :98
        const int byte_index = tail >> 3;
        if (len - head - byte_index + 2 < 0) return false;
        if (byte_index >= len) return false;                            // the reference would panic; needs len < 3
        if (tw_n == 0) refill();
        bit = (int)(tw & 1u);
        tw >>= 1;
        tw_n -= 1;
        tail += 1;
        return true;
    }
    // n (1 or 2) consecutive read_tail_bool calls at once: the bounds tests are monotonic in the bit position, so the
    // n calls all succeed exactly when the last one does, and a failure of any of them discards the frame anyway
    __device__ __forceinline__ bool tail_bools(int n, uint32_t& bits) {
        const int byte_index = (tail + n - 1) >> 3;
        if (len - head - byte_index + 2 < 0) return false;
        if (byte_index >= len) return false;
        if (tw_n < n) refill();
        bits = (uint32_t)tw & ((1u << n) - 1u);
        tw >>= n;
        tw_n -= n;
        tail += n;
        return true;
    }
    __device__ __forceinline__ bool tail_uint(int num_bits, uint32_t& out) {   // :63
        const int byte_index = tail >> 3, bit_index = tail & 7;
        const int add_bytes = (num_bits > 8 - bit_index && num_bits < 8) ? 2 : 1;
        const int num_bytes = (num_bits >> 3) + add_bytes;
        if (len - head - byte_index - num_bytes < 0) return false;
        // same value as the reference's big-endian load + shifts: the next num_bits bits, LSB first
        if (tw_n < num_bits) refill();
        out = (uint32_t)(tw & ((1ull << num_bits) - 1ull));
        tw >>= num_bits;
        tw_n -= num_bits;
        tail += num_bits;
        return true;
    }
};

struct AcState { uint32_t low, range; };

// Offset of line k in a thread's slice of the integer scratch xq[block32][k / 4][lane][k % 4] (int32 units, relative to
// the thread's base pointer, which already carries lane * 4).
__device__ __forceinline__ int xq_off(int k) { return (k >> 2) * 128 + (k & 3); }

// q = floor(low / tmp) for low < 2^24, 64 <= tmp < 2^14: the float quotient is within 1 of the truth, fix it up exactly
__device__ __forceinline__ uint32_t exact_quotient(uint32_t low, uint32_t tmp) {
    uint32_t q = (uint32_t)__fdividef((float)low, (float)tmp);
    int32_t r = (int32_t)(low - q * tmp);
    if (r < 0) q -= 1;
    else if ((uint32_t)r >= tmp) q += 1;
    return q;
}

// The spectral loop's version: min(floor(low / tmp), 1023) or 1024 with fewer integer-pipe operations.  low and tmp are
// exact in f32; the reciprocal estimate (relative error < 2^-21.4 after the multiply) scaled by 1 - 2^-20 lies below the
// true quotient by less than 0.002 whenever that quotient is below 1024, so its truncation is q or q - 1 and one
// upward fix-up suffices.  Quotients >= 1024 only occur on frames the caller has already marked bad.
__device__ __forceinline__ uint32_t quotient_spec(uint32_t low, uint32_t tmp) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"((float)tmp));
    uint32_t q = min((uint32_t)__fmul_rn(__fmul_rn((float)low, r), 0.99999904632568359375f), 1023u);
    if (low - q * tmp >= tmp) q += 1;
    return q;
}

__device__ __forceinline__ bool ac_finish(Reader& rd, AcState& st, uint32_t tmp, uint32_t e) {
    st.low -= tmp * (e & 0xffffu);
    st.range = tmp * (e >> 16);
    while (st.range < 0x10000u) {
        uint32_t b;
        if (!rd.head_byte(b)) return false;
        st.low = ((st.low << 8) & 0x00ffffffu) + b;
        st.range <<= 8;
    }
    return true;
}

// arithmetic_codec.rs:67-97.  `tab` holds cum | freq << 16 per symbol; the reference scans from the top for the
// largest val with tmp * cum[val] <= low, i.e. cum[val] <= floor(low / tmp).
__device__ __forceinline__ bool ac_decode(Reader& rd, AcState& st, const uint32_t* __restrict__ tab, int nsym, int& sym) {
    const uint32_t tmp = st.range >> 10;
    if (st.low >= (tmp << 10)) return false;                            // AcRangeFlOutOfRange
    const uint32_t q = exact_quotient(st.low, tmp);
    int val;
    if (nsym == 17) {
        val = ((tab[16] & 0xffffu) <= q) ? 16 : 0;
        if (val == 0) {
            if ((tab[8] & 0xffffu) <= q) val = 8;
            if ((tab[val + 4] & 0xffffu) <= q) val += 4;
            if ((tab[val + 2] & 0xffffu) <= q) val += 2;
            if ((tab[val + 1] & 0xffffu) <= q) val += 1;
        }
    } else {                                                            // 8 symbols (TNS order)
        val = 0;
        if ((tab[4] & 0xffffu) <= q) val = 4;
        if ((tab[val + 2] & 0xffffu) <= q) val += 2;
        if ((tab[val + 1] & 0xffffu) <= q) val += 1;
    }
    sym = val;
    return ac_finish(rd, st, tmp, tab[val]);
}

// Spectral symbols (decode_spectral_data below) answer the same search from shared memory: a coarse table gives the
// symbol at the start of the quotient's 32-wide bucket; the cumulative table (rows padded to SPEC_CF_STRIDE with
// 0xffff sentinels) is then walked upward three entries at a time - independent loads, and almost always one round.
constexpr int SPEC_CF_STRIDE = 20;

// mpvq_deenum, spectral_noise_shaping.rs:155-235.  y lives in shared memory (per-thread column).
__device__ void mpvq_deenum(int dim_in, int k_val_in, int ls_ind, uint32_t mpvq_ind, float* y, int ystride) {
    for (int i = 0; i < dim_in; i++) y[i * ystride] = 0.0f;
    int leading_sign = ls_ind == 0 ? 1 : -1;
    int k_max_local = k_val_in;
    uint32_t ind = mpvq_ind;
    for (int pos = 0; pos < dim_in; pos++) {
        const uint32_t* h_row = LC3T_MPVQ_OFFSETS[dim_in - 1 - pos];
        int k_delta;
        if (ind != 0) {
            int k_acc = k_max_local;
            uint32_t off = h_row[k_acc];
            bool wrap_flag = ind < off;
            uint32_t ul_diff = 0;
            if (!wrap_flag) ul_diff = ind - off;
            while (wrap_flag) {
                k_acc -= 1;
                wrap_flag = ind < h_row[k_acc];
                if (!wrap_flag) ul_diff = ind - h_row[k_acc];
            }
            ind = ul_diff;
            k_delta = k_max_local - k_acc;
        } else {
            y[pos * ystride] = (float)(leading_sign < 0 ? -k_max_local : k_max_local);
            break;
        }
        if (k_delta != 0) {
            y[pos * ystride] = (float)(leading_sign < 0 ? -k_delta : k_delta);
            leading_sign = (ind & 1) ? -1 : 1;
            ind >>= 1;
            k_max_local -= k_delta;
        }
    }
}

struct SideInfoD {
    int bw, lastnz, lsb_mode, gg_ind, num_tns, rc_in0, rc_in1;
    int ind_lf, ind_hf, ls_inda, ls_indb, idx_a, idx_b, submode_lsb, submode_msb, g_ind;
    int pitch_present, ltpf_active, pitch_index, noise_factor;
};

// side_info_reader.rs:29-200
__device__ bool read_side_info(Reader& rd, const DevConfig& c, SideInfoD& s) {
    uint32_t v;
    s.bw = 0;
    if (c.nbits_bw > 0) {
        if (!rd.tail_uint(c.nbits_bw, v)) return false;
        if ((uint32_t)c.fs_ind < v) return false;
        s.bw = (int)v;
    }
    if (!rd.tail_uint(c.lastnz_bits, v)) return false;
    s.lastnz = (int)((v + 1) << 1);
    if (s.lastnz > c.ne) return false;
    if (!rd.tail_bool(s.lsb_mode)) return false;
    if (!rd.tail_uint(8, v)) return false;
    s.gg_ind = (int)v;
    s.num_tns = s.bw < 3 ? 1 : 2;
    s.rc_in0 = s.rc_in1 = 0;
    if (!rd.tail_bool(s.rc_in0)) return false;
    if (s.num_tns == 2 && !rd.tail_bool(s.rc_in1)) return false;
    if (!rd.tail_bool(s.pitch_present)) return false;
    // read_sns_vq :127
    if (!rd.tail_uint(5, v)) return false;
    s.ind_lf = (int)v;
    if (!rd.tail_uint(5, v)) return false;
    s.ind_hf = (int)v;
    if (!rd.tail_bool(s.submode_msb)) return false;
    if (!rd.tail_uint(s.submode_msb == 0 ? 1 : 2, v)) return false;
    int g_ind = (int)v;
    if (!rd.tail_bool(s.ls_inda)) return false;
    if (s.submode_msb == 0) {
        if (!rd.tail_uint(25, v)) return false;
        if (v >= 33460056u) return false;
        int idx_bor = (int)(v / 2390004u);
        s.idx_a = (int)(v - (uint32_t)idx_bor * 2390004u);
        s.submode_lsb = 0;
        int t = idx_bor - 2;
        if (t < 0) s.submode_lsb = 1;
        int u = t + s.submode_lsb * 2;
        if (s.submode_lsb != 0) { g_ind = (g_ind << 1) + u; s.idx_b = 0; s.ls_indb = 0; }
        else { s.idx_b = u >> 1; s.ls_indb = u & 1; }
    } else {
        s.ls_indb = 0; s.idx_b = 0; s.submode_lsb = 0;
        if (!rd.tail_uint(24, v)) return false;
        if (v >= 16708096u) return false;
        if (v >= 15158272u) {
            v -= 15158272u;
            s.submode_lsb = 1;
            g_ind = (g_ind << 1) + (int)(v & 1);
            s.idx_a = (int)(v >> 1);
        } else s.idx_a = (int)v;
    }
    s.g_ind = g_ind;
    s.ltpf_active = 0;
    s.pitch_index = 0;
    if (s.pitch_present) {
        if (!rd.tail_bool(s.ltpf_active)) return false;
        if (!rd.tail_uint(9, v)) return false;
        s.pitch_index = (int)v;
    }
    if (!rd.tail_uint(3, v)) return false;
    s.noise_factor = (int)v;
    return true;
}

constexpr int ENT_THREADS = 128;

// Stage the CTA's frames into shared-memory rows (odd word pitch).  Dense input (frame_stride == nbytes, 16-byte
// aligned block) is fetched with 16-byte loads and scattered byte by byte; otherwise byte by byte from the start.
__device__ __forceinline__ void stage_rows(const EntropyParams& p, uint8_t* s_rows, int stream0, int tid) {
    const int n_rows = min(ENT_THREADS, p.n_streams - stream0);
    const int nb = p.nbytes;
    const int total = n_rows * nb;
    const uint8_t* src = p.frames + (size_t)stream0 * p.frame_stride;
    int done = 0;
    if (p.frame_stride == (size_t)nb && (((uintptr_t)src) & 15) == 0) {
        const int n16 = total >> 4;
        for (int i = tid; i < n16; i += ENT_THREADS) {
            const uint4 v = ((const uint4*)src)[i];
            const uint32_t w[4] = {v.x, v.y, v.z, v.w};
            int r = (16 * i) / nb, b = 16 * i - r * nb;
#pragma unroll
            for (int j = 0; j < 16; j++) {
                s_rows[r * p.row_pitch + b] = (uint8_t)(w[j >> 2] >> (8 * (j & 3)));
                if (++b == nb) { b = 0; r++; }
            }
        }
        done = n16 << 4;
    }
    for (int i = done + tid; i < total; i += ENT_THREADS) {
        const int r = i / nb, b = i - r * nb;
        s_rows[r * p.row_pitch + b] = src[(size_t)r * p.frame_stride + b];
    }
}

// Hand-off record entropy_kernel -> dequant_kernel, one per THREAD SLOT (stream0 + tid) because the integer spectrum
// sits in that thread's lane-interleaved scratch column; HO_FID names the frame (row of the CTA) the slot decoded.
enum {
    HO_OK = 0, HO_FID, HO_LASTNZ, HO_LSB_MODE, HO_GG_IND, HO_BW, HO_NUM_TNS, HO_NOISE_FACTOR, HO_RC_ORDER0, HO_RC_ORDER1,
    HO_IND_LF, HO_IND_HF, HO_SUBMODE_MSB, HO_SUBMODE_LSB, HO_G_IND, HO_LS_INDA, HO_LS_INDB, HO_IDX_A, HO_IDX_B,
    HO_NRES, HO_SEED, HO_TAIL, HO_HEAD, HO_LEN, HO_LTPF_ACTIVE, HO_PITCH_INDEX, HO_PAD0, HO_PAD1,
    HO_RC_I = 28
};
static_assert(HO_RC_I + 16 == HO_WORDS, "hand-off record size");

// shared-memory carve-ups (bytes), T = ENT_THREADS
// entropy_kernel:
//   lookup  4096            AC_SPEC_LOOKUP
//   clut    2048            coarse symbol table (64 models x 32 quotient buckets)
//   spec_cf 64*20*4         cum | freq << 16, rows padded with sentinels
//   tns_cf  (2*8 + 8*17)*4  order tables then coef tables
//   lev     7*T*4           lsb-mode save_lev flags, one bit per tuple
//   sort    2*T*4           work-sorting keys and the resulting frame assignment
//   rows    T*row_pitch     staged frame bytes
// dequant_kernel:
//   scf     16*T*4          per-thread SNS scale factors (also the PVQ vector while de-enumerating)
//   band    68*4            I_fs band edges
//   rows    T*row_pitch     staged frame bytes (residual bits)
__host__ __device__ inline size_t entropy_smem_bytes(int row_pitch) {
    return 4096 + 2048 + 64 * 20 * 4 + (2 * 8 + 8 * 17) * 4 + 7 * ENT_THREADS * 4 + 2 * ENT_THREADS * 4 + (size_t)ENT_THREADS * row_pitch;
}
__host__ __device__ inline size_t dequant_smem_bytes(int row_pitch) {
    return 16 * ENT_THREADS * 4 + 68 * 4 + (size_t)ENT_THREADS * row_pitch;
}

template <bool IDS>
__device__ __forceinline__ void entropy_body(const EntropyParams& p, const int block) {
    // declared here, not handed in as a pointer: the compiler then addresses shared memory directly instead of rebuilding the
    // shared window base from a generic pointer inside the symbol loop
    extern __shared__ __align__(16) uint8_t smem[];
    uint8_t* s_lookup = smem;
    uint8_t* s_clut = smem + 4096;
    uint32_t* s_spec_cf = (uint32_t*)(smem + 4096 + 2048);
    uint32_t* s_tns_cf = s_spec_cf + 64 * SPEC_CF_STRIDE;
    uint32_t* s_lev = s_tns_cf + (2 * 8 + 8 * 17);
    int32_t* s_key = (int32_t*)(s_lev + 7 * ENT_THREADS);
    int32_t* s_owner = s_key + ENT_THREADS;
    uint8_t* s_rows = (uint8_t*)(s_owner + ENT_THREADS);

    const DevConfig& c = *p.cfg;
    const int tid = threadIdx.x, lane = tid & 31;
    const int stream0 = block * ENT_THREADS;
    const int ne = c.ne;

    // ---- stage tables and frame bytes
    for (int i = tid; i < 4096 / 4; i += ENT_THREADS) ((uint32_t*)s_lookup)[i] = ((const uint32_t*)LC3T_AC_SPEC_LOOKUP)[i];
    for (int i = tid; i < 2048 / 4; i += ENT_THREADS) ((uint32_t*)s_clut)[i] = ((const uint32_t*)p.sym_lut)[i];
    for (int i = tid; i < 64 * SPEC_CF_STRIDE; i += ENT_THREADS) {
        const int pk = i / SPEC_CF_STRIDE, j = i - pk * SPEC_CF_STRIDE;
        s_spec_cf[i] = j < 17 ? ((uint32_t)(uint16_t)LC3T_AC_SPEC_CUMFREQ[pk][j] | ((uint32_t)(uint16_t)LC3T_AC_SPEC_FREQ[pk][j] << 16)) : 0xffffu;
    }
    for (int i = tid; i < 2 * 8; i += ENT_THREADS)
        s_tns_cf[i] = (uint32_t)(uint16_t)(&LC3T_AC_TNS_ORDER_CUMFREQ[0][0])[i] | ((uint32_t)(uint16_t)(&LC3T_AC_TNS_ORDER_FREQ[0][0])[i] << 16);
    for (int i = tid; i < 8 * 17; i += ENT_THREADS)
        s_tns_cf[16 + i] = (uint32_t)(uint16_t)(&LC3T_AC_TNS_COEF_CUMFREQ[0][0])[i] | ((uint32_t)(uint16_t)(&LC3T_AC_TNS_COEF_FREQ[0][0])[i] << 16);
    for (int i = tid; i < 7 * ENT_THREADS; i += ENT_THREADS) s_lev[i] = 0;
    {
        stage_rows(p, s_rows, stream0, tid);
    }
    __syncthreads();

    // ---- work sorting: the spectral loop runs one iteration per arithmetic symbol (lastnz/2 tuples plus their escape
    // levels), which varies widely between streams.  Frames of the CTA are handed to threads in order of decreasing
    // expected work so that the 32 lanes of a warp finish together (frames live in shared rows, so any thread can take
    // any frame; per-thread scratch stays indexed by tid).  The predictor is the number of symbols the stream's PREVIOUS
    // good frame took (audio is stationary over a frame: correlation 0.91 on the corpus, lanes busy 80 % of a warp's
    // iterations); a stream without history falls back to lastnz from the side information (correlation 0.37, 70 %).
    // Two flags of the side information class the frames first, because they switch on code only a few lanes run:
    //   lsb_mode (7 % of frames: the refinement pass after the spectral loop) - these frames lead, so one warp of the
    //     CTA walks that pass with several lanes instead of all four with one or two;
    //   an active TNS filter (43 %: the TNS symbols here, the lattice in dequant_kernel, which runs at the warp's largest
    //     order) - frames with TNS follow in decreasing order of work, frames without it close in INCREASING order, so
    //     that the warp holding the class boundary gets the light frames of both sides.
    // On the bench corpus: warps walking the refinement pass 88 % -> 25 %, warps running the lattice 93 % -> 52 %, for
    // 3 % more iterations of the spectral loop.
    {
        int key = -1;
        const int s_me = stream0 + tid;
        if (s_me < p.n_streams) {
            int len = p.frame_nbytes ? p.frame_nbytes[s_me] : p.nbytes;
            len = min(max(len, 0), p.nbytes);
            if (len < p.min_nbytes) len = 0;
            Reader pr;
            pr.buf = s_rows + tid * p.row_pitch;
            pr.len = len; pr.head = 0; pr.tail = 0; pr.tw = 0; pr.tw_n = 0;
            uint32_t v = 0, bwv = 0;
            key = 0;
            bool good = true;
            if (c.nbits_bw > 0) { good = pr.tail_uint(c.nbits_bw, v); bwv = v; }
            if (good && pr.tail_uint(c.lastnz_bits, v)) {
                int work = (int)((v + 1) << 1);
                if (p.nsym_prev) {
                    const int prev = p.nsym_prev[state_row<IDS>(p.ids, s_me)];
                    if (prev > 0) work = prev;
                }
                work = min(work, 0xffff);
                uint32_t fl = 0;                                        // lsb_mode, 8 bits of gain, rc_order flags
                int cls = 1;
                if (pr.tail_uint(bwv < 3 ? 10 : 11, fl)) cls = (fl & 1u) ? 3 : ((fl >> 9) != 0u ? 2 : 1);
                key = cls == 1 ? (1 << 16) + (0xffff - work) : (cls << 16) + work;
            }
        }
        s_key[tid] = key;
        __syncthreads();
        int rank = 0;
        for (int u = 0; u < ENT_THREADS; u++) {
            const int ku = s_key[u];
            rank += (ku > key) || (ku == key && u < tid);
        }
        s_owner[rank] = tid;
        __syncthreads();
    }
    const int fid = s_owner[tid];                                      // frame (row) of this CTA handled by this thread
    const int stream = stream0 + fid;
    const bool live = stream < p.n_streams;

    // ---- per-frame serial decode (pass 1)
    Reader rd;
    rd.buf = s_rows + fid * p.row_pitch;
    rd.len = live ? (p.frame_nbytes ? p.frame_nbytes[stream] : p.nbytes) : 0;
    if (rd.len > p.nbytes) rd.len = p.nbytes;
    if (rd.len < 0) rd.len = 0;
    if (rd.len < p.min_nbytes) rd.len = 0;                              // shorter than the handle's promised minimum: treated as lost
    rd.head = 0;
    rd.tail = 0;
    rd.tw = 0;
    rd.tw_n = 0;
    const int nbits = rd.len * 8;
    int32_t* xq = p.xq + ((size_t)((stream0 + tid) >> 5) * ne) * 32 + lane * 4;   // thread-private slice, line k at xq[xq_off(k)]

    SideInfoD si;
    bool ok = live && read_side_info(rd, c, si);
    int rc_order0 = 0, rc_order1 = 0;
    int rc_i[16];
#pragma unroll
    for (int i = 0; i < 16; i++) rc_i[i] = 0;
    AcState ac{0, 0x00ffffffu};
    uint32_t seed_acc = 0;     // sum |x_k| * k, wrapping (arithmetic_codec.rs:140-145)
    int nres = 0;

    if (ok) {                                                          // ac_dec_init :57
        if (rd.head + 2 < rd.len) {
            ac.low = ((uint32_t)rd.buf[0] << 16) | ((uint32_t)rd.buf[1] << 8) | rd.buf[2];
            rd.head = 3;
        } else ok = false;
    }
    if (ok) {                                                          // decode_tns_data :307
        const int max_bits = c.n_ms == LC3B_7P5MS ? 360 : 480;
        const int w = nbits < max_bits ? 1 : 0;
        rc_order0 = si.rc_in0;
        rc_order1 = si.rc_in1;
#pragma unroll
        for (int f = 0; f < 2; f++) {
            int& ord = f == 0 ? rc_order0 : rc_order1;
            if (ok && f < si.num_tns && ord > 0) {
                int o;
                ok = ac_decode(rd, ac, s_tns_cf + w * 8, 8, o);
                if (ok) {
                    ord = o + 1;
#pragma unroll
                    for (int k = 0; k < 8; k++) {
                        if (ok && k < ord) {
                            int sym;
                            ok = ac_decode(rd, ac, s_tns_cf + 16 + k * 17, 17, sym);
                            rc_i[f * 8 + k] = sym;
                        }
                    }
                }
            }
        }
    }
    if (ok) {                                                          // decode_spectral_data :211
        // One arithmetic symbol per iteration for every lane (escape or final), instead of a per-tuple inner loop:
        // lanes sit at different tuples/levels but all execute the same decode.  The body is straight-line code:
        // renormalisation, the tail bits of the symbol (escape magnitude bits and/or signs, at most 4, peeked from
        // the staged row without a bit window to refill) and the tuple bookkeeping are selects, and every failure
        // of the reference's readers sets a sticky flag that ends the lane's loop - a frame that fails anywhere is
        // discarded whole, so when exactly the flag is acted on does not matter.
        const int rate_flag = nbits > (160 + c.fs_ind * 160) ? 512 : 0;
        const int half_ne = ne / 2;
        const uint8_t* buf = rd.buf;
        const int len = rd.len;
        int head = rd.head, tail = rd.tail;
        uint32_t low = ac.low, range = ac.range;
        int ctx = 0;
        const int ntup = si.lastnz >> 1;
        int k = 0, lev = 0, xa_ = 0, xb_ = 0;
        uint32_t lev_word = 0;                                          // save_lev flags of the current 32 tuples
        bool bad = false;
        int nsym = 0;                                                   // iterations = arithmetic symbols of this frame
        while (k < ntup && !bad) {
            nsym++;
            const int t0 = ctx + rate_flag + ((k * 2) > half_ne ? 256 : 0);
            const int pki = s_lookup[t0 + min(lev, 3) * 1024];
            const uint32_t* tab = s_spec_cf + pki * SPEC_CF_STRIDE;
            // ac_decode :67-97
            const uint32_t tmp = range >> 10;
            bad |= low >= (tmp << 10);                                  // AcRangeFlOutOfRange
            const uint32_t q = quotient_spec(low, tmp);
            int val = s_clut[pki * 32 + (q >> 5)];
            for (;;) {                                                  // almost always a single round
                const uint32_t c1 = tab[val + 1] & 0xffffu, c2 = tab[val + 2] & 0xffffu, c3 = tab[val + 3] & 0xffffu;
                const int adv = (int)(c1 <= q) + (int)(c2 <= q) + (int)(c3 <= q);   // cum is non-decreasing
                val += adv;
                if (!__any_sync(__activemask(), adv == 3)) break;
            }
            const uint32_t e = tab[val];
            low -= tmp * (e & 0xffffu);
            range = tmp * (e >> 16);
            {   // renormalisation: range >= 64 here, so at most two bytes
                const int nsh = (int)(range < 0x10000u) + (int)(range < 0x100u);
                const uint32_t b0 = buf[head], b1 = buf[head + 1];
                const uint32_t in = nsh == 2 ? ((b0 << 8) | b1) : b0;
                low = nsh ? (((low << (8 * nsh)) & 0x00ffffffu) + in) : low;
                range <<= 8 * nsh;
                head += nsh;
                bad |= head > len;                                      // read_head_byte past the end
            }
            // the next tail bits, LSB first (buffer_reader.rs:98): 9 usable bits after the in-byte shift
            uint32_t w;
            {
                const int i0 = len - 1 - (tail >> 3);
                const uint32_t y0 = buf[max(i0, 0)], y1 = buf[max(i0 - 1, 0)];
                w = (y0 | (y1 << 8)) >> (tail & 7);
            }
            const bool esc = val >= 16;
            const bool esc_bits = esc && (!si.lsb_mode || lev > 0);     // escape: two more magnitude bits
            const uint32_t eb = esc_bits ? (w & 3u) : 0u;
            const int n_esc = esc_bits ? 2 : 0;
            xa_ += (int)(eb & 1u) << lev;
            xb_ += (int)(eb >> 1) << lev;
            const int lev2 = lev + (esc ? 1 : 0);
            const bool fin = !esc || lev2 >= 14;                        // QUIRK (ii): at lev == 14 the tuple ends with sym == 16
            const int a = val & 3, b = val >> 2;
            if (fin) { xa_ += a << lev2; xb_ += b << lev2; }
            const int nsign = fin ? (int)(xa_ > 0) + (int)(xb_ > 0) : 0;
            const int nrd = n_esc + nsign;
            if (nrd > 0) {                                              // bounds of the last read_tail_bool (:98-103)
                const int byte_index = (tail + nrd - 1) >> 3;
                bad |= (len - head - byte_index + 2 < 0) || (byte_index >= len);
            }
            tail += nrd;
            uint32_t sg = w >> n_esc;
            if (fin) {
                if (xa_ > 0) { xa_ = (sg & 1u) ? -xa_ : xa_; sg >>= 1; }
                if (xb_ > 0) xb_ = (sg & 1u) ? -xb_ : xb_;
                if (!bad) {
                    *(int2*)(xq + xq_off(2 * k)) = make_int2(xa_, xb_);   // lines 2k, 2k + 1 share a 16-byte group
                }
                seed_acc += (uint32_t)abs(xa_) * (uint32_t)(2 * k) + (uint32_t)abs(xb_) * (uint32_t)(2 * k + 1);
                lev_word |= (si.lsb_mode && lev2 > 0) ? (1u << (k & 31)) : 0u;   // save_lev[k], QUIRK (i)
                if ((k & 31) == 31 || k == ntup - 1) { s_lev[(k >> 5) * ENT_THREADS + tid] = lev_word; lev_word = 0; }
                const int l = min(lev2, 3);
                const int t1 = (l <= 1) ? 1 + (a + b) * (l + 1) : 12 + l;
                ctx = (ctx & 15) * 16 + t1;
                k++;
                xa_ = 0;
                xb_ = 0;
            }
            lev = fin ? 0 : lev2;
        }
        ok = !bad;
        if (ok && p.nsym_prev) p.nsym_prev[state_row<IDS>(p.ids, stream)] = nsym;   // next frame's sort key
        ac.low = low;
        ac.range = range;
        rd.head = head;
        rd.tail = tail;
        {   // resume the windowed tail reader mid-byte: (tail + tw_n) % 8 == 0
            const int idx = len - 1 - (tail >> 3);
            const uint32_t byte = (idx >= 0 && idx < len) ? buf[idx] : 0u;
            rd.tw = (uint64_t)(byte >> (tail & 7));
            rd.tw_n = 8 - (tail & 7);
        }
    }
    if (ok) {                                                          // calc_num_residual_bits :390
        const int nbits_side = rd.tail - 8;
        const int nbits_ari = (rd.head + 1 - 3) * 8 + 25 - (31 - __clz(ac.range));
        if (nbits < nbits_side + nbits_ari) ok = false;                 // NegativeResidualNumBits
        nres = nbits - nbits_side - nbits_ari;
    }
    if (ok && si.lsb_mode) {                                           // decode_residual_bits (lsb branch) :193-207
        // QUIRK (i): flags were stored per TUPLE index but are consumed per LINE index k = 0, 2, 4, ...
        int left = nres;
        bool stop = false;
        // save_lev[] is only ever written for tuple indices < lastnz/2 and is zero beyond, so the walk can stop there.
        for (int k = 0; k < (si.lastnz >> 1) && !stop; k += 2) {
            if (!((s_lev[(k >> 5) * ENT_THREADS + tid] >> (k & 31)) & 1u)) continue;
            // lines k and k + 1 (k even) are one 8-byte half of a group: one load, one store, instead of a dependent
            // round trip to L2 per refined line
            int2 vv = *(const int2*)(xq + xq_off(k));
            bool touched = false;
#pragma unroll
            for (int j = 0; j < 2; j++) {                               // read_res_bit :346
                if (stop) break;
                if (left == 0) { stop = true; break; }
                int bit;
                if (!rd.tail_bool(bit)) { ok = false; stop = true; break; }
                left--;
                if (bit) {
                    const int idx = k + j;
                    int v = j == 0 ? vv.x : vv.y;
                    if (v > 0) { v += 1; seed_acc += (uint32_t)idx; }
                    else if (v < 0) { v -= 1; seed_acc += (uint32_t)idx; }
                    else {
                        if (left == 0) { stop = true; break; }
                        if (!rd.tail_bool(bit)) { ok = false; stop = true; break; }
                        left--;
                        v = bit ? -1 : 1;
                        seed_acc += (uint32_t)idx;
                    }
                    if (j == 0) vv.x = v; else vv.y = v;
                    touched = true;
                }
            }
            if (touched) *(int2*)(xq + xq_off(k)) = vv;
        }
    }

    // ---- hand-off to dequant_kernel, status, inspection
    {
        int32_t* ho = p.handoff + (size_t)(stream0 + tid) * HO_WORDS;
        ho[HO_OK] = ok; ho[HO_FID] = fid;
        ho[HO_LASTNZ] = si.lastnz; ho[HO_LSB_MODE] = si.lsb_mode; ho[HO_GG_IND] = si.gg_ind; ho[HO_BW] = si.bw;
        ho[HO_NUM_TNS] = si.num_tns; ho[HO_NOISE_FACTOR] = si.noise_factor; ho[HO_RC_ORDER0] = rc_order0; ho[HO_RC_ORDER1] = rc_order1;
        ho[HO_IND_LF] = si.ind_lf; ho[HO_IND_HF] = si.ind_hf; ho[HO_SUBMODE_MSB] = si.submode_msb; ho[HO_SUBMODE_LSB] = si.submode_lsb;
        ho[HO_G_IND] = si.g_ind; ho[HO_LS_INDA] = si.ls_inda; ho[HO_LS_INDB] = si.ls_indb; ho[HO_IDX_A] = si.idx_a; ho[HO_IDX_B] = si.idx_b;
        ho[HO_NRES] = nres; ho[HO_SEED] = (int32_t)seed_acc; ho[HO_TAIL] = rd.tail; ho[HO_HEAD] = rd.head; ho[HO_LEN] = rd.len;
        ho[HO_LTPF_ACTIVE] = si.ltpf_active; ho[HO_PITCH_INDEX] = si.pitch_index;
#pragma unroll
        for (int i = 0; i < 16; i++) ho[HO_RC_I + i] = rc_i[i];
    }
    if (live) {
        if (p.status_out) p.status_out[stream] = ok ? 0 : 1;
        if (p.trace) {
            const bool is_zero_frame = ok && si.lastnz == 2 && xq[0] == 0 && xq[1] == 0 && si.gg_ind == 0;
            int32_t* tr = p.trace + (size_t)stream * LC3B_TRACE_WORDS;
            for (int i = 0; i < LC3B_TRACE_WORDS; i++) tr[i] = 0;
            tr[LC3B_TR_OK] = ok;
            if (ok) {
                tr[LC3B_TR_BW] = si.bw; tr[LC3B_TR_LASTNZ] = si.lastnz; tr[LC3B_TR_LSB_MODE] = si.lsb_mode;
                tr[LC3B_TR_GG_IND] = si.gg_ind; tr[LC3B_TR_NUM_TNS] = si.num_tns; tr[LC3B_TR_RC_ORDER_IN0] = si.rc_in0;
                tr[LC3B_TR_RC_ORDER_IN1] = si.rc_in1; tr[LC3B_TR_IND_LF] = si.ind_lf; tr[LC3B_TR_IND_HF] = si.ind_hf;
                tr[LC3B_TR_LS_INDA] = si.ls_inda; tr[LC3B_TR_LS_INDB] = si.ls_indb; tr[LC3B_TR_IDX_A] = si.idx_a;
                tr[LC3B_TR_IDX_B] = si.idx_b; tr[LC3B_TR_SUBMODE_LSB] = si.submode_lsb; tr[LC3B_TR_SUBMODE_MSB] = si.submode_msb;
                tr[LC3B_TR_G_IND] = si.g_ind; tr[LC3B_TR_PITCH_PRESENT] = si.pitch_present; tr[LC3B_TR_LTPF_ACTIVE] = si.ltpf_active;
                tr[LC3B_TR_PITCH_INDEX] = si.pitch_index; tr[LC3B_TR_NOISE_FACTOR] = si.noise_factor;
                tr[LC3B_TR_RC_ORDER0] = rc_order0; tr[LC3B_TR_RC_ORDER1] = rc_order1;
#pragma unroll
                for (int i = 0; i < 16; i++) tr[LC3B_TR_RC_I0 + i] = rc_i[i];
                // residual_bits.len(): bits actually consumed in the non-lsb branch, 0 in lsb mode (:160-209)
                int n_nonzero_used = 0;
                if (!si.lsb_mode) {
                    int cnt = 0;
                    for (int k = 0; k < si.lastnz && cnt < nres; k++) if (xq[xq_off(k)] != 0) cnt++;
                    n_nonzero_used = cnt;
                }
                tr[LC3B_TR_NRES] = n_nonzero_used;
                tr[LC3B_TR_SEED] = (int32_t)(seed_acc & 0xffffu);
                tr[LC3B_TR_IS_ZERO] = is_zero_frame;
            }
        }
        if (p.trace_x) {
            int32_t* tx = p.trace_x + (size_t)stream * ne;
            for (int k = 0; k < ne; k++) tx[k] = (ok && k < si.lastnz) ? xq[xq_off(k)] : 0;
        }
    }
}


template <bool IDS>
__global__ void __launch_bounds__(ENT_THREADS, 6) entropy_kernel(const __grid_constant__ EntropyParams p) {
    entropy_body<IDS>(p, blockIdx.x);
}

// Mixed-rate batches (BASELINE config 4; lc3b_mixed_*): ONE launch covers every (fs, duration) bucket.  A CTA finds its
// bucket in a small device table, patches the per-call pointers into that bucket's parameter block (rows of the caller's
// buffers are in bucket order, so a bucket is a contiguous row range) and runs the single-configuration body on it.
// per_entropy_cta: CTAs of the calling kernel per entropy CTA of ENT_THREADS thread slots (a bucket's first_cta counts
// entropy CTAs): 1 but for the warp-per-frame kernel, whose CTAs cover DQW_WARPS slots.
__device__ __forceinline__ void mixed_select(const MixedParams& m, EntropyParams* s_p, int* s_block, int per_entropy_cta) {
    if (threadIdx.x == 0) {
        int b = 0;
        while (b + 1 < m.n_buckets && (int)blockIdx.x >= m.buckets[b + 1].first_cta * per_entropy_cta) b++;
        const MixedBucket& bk = m.buckets[b];
        EntropyParams q = bk.ep;
        q.frames = m.frames + (size_t)bk.first_row * m.frame_stride;
        q.frame_nbytes = m.frame_nbytes ? m.frame_nbytes + bk.first_row : nullptr;
        q.nbytes = m.nbytes;
        q.frame_stride = m.frame_stride;
        q.status_out = m.status_out ? m.status_out + bk.first_row : nullptr;
        q.row_pitch = m.row_pitch;
        *s_p = q;
        *s_block = (int)blockIdx.x - bk.first_cta * per_entropy_cta;
    }
    __syncthreads();
}

__global__ void __launch_bounds__(ENT_THREADS, 6) entropy_mixed_kernel(const __grid_constant__ MixedParams m) {
    __shared__ EntropyParams s_p;
    __shared__ int s_block;
    mixed_select(m, &s_p, &s_block, 1);
    entropy_body<false>(s_p, s_block);
}

// ---------------------------------------------------------------- reference steps D4-D8, one definition each
// Shared by the thread-per-frame (dequant_body), warp-per-frame (dequant_warp_body) and lattice (tns_list_body) kernels,
// so that the kernels' f32 operations are the same ones in the same order and their spectra are bit-identical.

__device__ __forceinline__ int bw_stop_lines(const DevConfig& c, int bw) {
    return c.n_ms == LC3B_10MS ? 80 * (bw + 1) : 60 * (bw + 1);
}

// Per-frame scalars: global gain (global_gain.rs:15-25), noise-filling level and the noise-filled line range.
struct FrameScalars {
    float gg, nf_level;
    int bw_stop, nf_start;
};
__device__ __forceinline__ FrameScalars frame_scalars(const DevConfig& c, int nbits, int gg_ind, int noise_factor, int bw) {
    FrameScalars f;
    const int fs = c.fs_ind + 1;
    const int gg_off = -min(nbits / (10 * fs), 115) - 105 - 5 * fs;
    f.gg = c.gg_table[gg_ind + gg_off + 245];
    f.nf_level = xd(xs(8.0f, (float)noise_factor), 16.0f);
    f.bw_stop = bw_stop_lines(c, bw);
    f.nf_start = c.n_ms == LC3B_10MS ? 24 : 18;
    return f;
}

// residual_spectrum.rs:13-39: non-zero line x refined by one tail bit
__device__ __forceinline__ float residual_refine(float v, int32_t xi, uint32_t bit) {
    const float up = xi > 0 ? 0.3125f : 0.1875f, down = xi > 0 ? -0.1875f : -0.3125f;
    return xa(v, bit ? up : down);
}

// noise_filling.rs:37-55: the level a filled line takes from the LCG state that filled it
__device__ __forceinline__ float nf_fill_level(uint32_t state, float nf_level) {
    return state < 0x8000u ? nf_level : -nf_level;
}
// one LCG step for a filled line; v passes through unchanged when the line is not filled
__device__ __forceinline__ float noise_fill(bool fill, int& nf_state, float nf_level, float v) {
    const int nxt = (13849 + nf_state * 31821) & 0xFFFF;
    nf_state = fill ? nxt : nf_state;
    return fill ? nf_fill_level((uint32_t)nxt, nf_level) : v;
}

// temporal_noise_shaping.rs:83-138: filter 0 runs over lines [s0, e0), filter 1 over [e0, e1) (empty below bw 3);
// ord1 is 0 for a frame with one filter.  rc_i: the 16 coefficient indices (an array or a hand-off pointer).
struct TnsPlan {
    float rc0[8], rc1[8];
    int ord0, ord1, s0, e0, e1;
};
template <typename RcIndices>
__device__ __forceinline__ void tns_plan(TnsPlan& f, const DevConfig& c, int bw, int num_tns, int order0, int order1,
                                         const RcIndices& rc_i) {
    const int bw_stop = bw_stop_lines(c, bw);
    f.s0 = c.n_ms == LC3B_10MS ? 12 : 9;
    if (bw < 3) { f.e0 = bw_stop; f.e1 = bw_stop; }
    else { f.e0 = bw_stop / 2; f.e1 = bw_stop; }
    f.ord0 = order0;
    f.ord1 = num_tns == 2 ? order1 : 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {                                       // QUIRK: index 0 -> rc = 0.0
        const int a = rc_i[i], b = rc_i[8 + i];
        f.rc0[i] = a != 0 ? c.tns_sin[a] : 0.0f;
        f.rc1[i] = b != 0 ? c.tns_sin[b] : 0.0f;
    }
}

// The filter change at line `next`: phase 0 -> 1 enters filter 0, 1 -> 2 filter 1 when it covers any line, and the end
// of the last filter sets the order to 0.  QUIRK: st is not reset, the lattice state carries across filters.
__device__ __forceinline__ void tns_switch(const TnsPlan& f, float (&rc)[8], int& ord, int& phase, int& next) {
    if (phase == 0) {
#pragma unroll
        for (int i = 0; i < 8; i++) rc[i] = f.rc0[i];
        ord = f.ord0;
        phase = 1;
        next = f.e0;
    } else if (phase == 1 && f.e0 < f.e1) {
#pragma unroll
        for (int i = 0; i < 8; i++) rc[i] = f.rc1[i];
        ord = f.ord1;
        phase = 2;
        next = f.e1;
    } else {
        ord = 0;
        next = 0x7fffffff;
    }
}

// temporal_noise_shaping.rs:24-74: one line through the all-pole lattice of order ord.  Lanes of a warp sit in different
// filters with different orders: the lattice runs `depth` stages (warp-uniform, at least the warp's largest order; a
// compile-time constant where the caller has one) and the stages at or above the lane's own order are selects that keep
// its value and state, so the warp never splits over it.
__device__ __forceinline__ float tns_lattice_line(float v, const float (&rc)[8], float (&st)[8], int ord, int depth) {
    if (depth <= 0) return v;
    float t = v;
#pragma unroll
    for (int j = 7; j >= 0; j--) {
        if (j < depth) {
            const float t2 = xs(t, xm(rc[j], st[j]));
            t = j < ord ? t2 : t;
            if (j + 1 < 8) {
                const float s2 = xa(xm(rc[j], t), st[j]);
                st[j + 1 < 8 ? j + 1 : 7] = j + 1 < ord ? s2 : st[j + 1 < 8 ? j + 1 : 7];
            }
        }
    }
    st[0] = ord > 0 ? t : st[0];
    return t;
}

// spectral_noise_shaping.rs:61-84: the shape vector (stride ys) into y and its gain divided by the vector's norm
__device__ __forceinline__ float sns_norm_gain(const float* yv, int ys, const float* gains, int g_ind, float (&y)[16]) {
    float sum = 0.0f;
#pragma unroll
    for (int i = 0; i < 16; i++) { y[i] = yv[i * ys]; sum = xa(sum, xm(y[i], y[i])); }
    const float y_norm = sqrtf(sum);
    float g = gains[g_ind];
    if (y_norm != 0.0f) g = xd(g, y_norm);
    return g;
}
// scale factor n: stage-1 codebook entry plus the gain times row n of the DCT rotation
__device__ __forceinline__ float sns_scale_factor(const float (&y)[16], float g, int n, int ind_lf, int ind_hf) {
    float factor = 0.0f;
#pragma unroll
    for (int col = 0; col < 16; col++) factor = xa(factor, xm(y[col], LC3T_D[n][col]));
    const float st1 = n < 8 ? LC3T_LFCB[ind_lf][n] : LC3T_HFCB[ind_hf][n - 8];
    return xa(st1, xm(g, factor));
}

// spectral_noise_shaping.rs:85-98: interpolated scale factor j of 64 from the 16 at scf[n * STRIDE]
template <int STRIDE>
__device__ __forceinline__ float sns_interp64(const float* scf, int j) {
    if (j < 2) return scf[0];
    if (j >= 62) {
        const float d = xs(scf[15 * STRIDE], scf[14 * STRIDE]);
        return xa(scf[15 * STRIDE], xm(j == 62 ? 0.125f : 0.375f, d));
    }
    const int n = (j - 2) >> 2, r = (j - 2) & 3;
    const float fn = scf[n * STRIDE], d = xs(scf[(n + 1) * STRIDE], fn);
    const float w = r == 0 ? 0.125f : r == 1 ? 0.375f : r == 2 ? 0.625f : 0.875f;
    return xa(fn, xm(w, d));
}
// :100-123: the gain of band b, the 64 interpolated values folded onto nb < 64 bands
template <int STRIDE>
__device__ __forceinline__ float sns_band_gain(const float* scf, int b, int nb) {
    const int n2 = 64 - nb;
    float s;
    if (n2 != 0) s = b < n2 ? xd(xa(sns_interp64<STRIDE>(scf, 2 * b), sns_interp64<STRIDE>(scf, 2 * b + 1)), 2.0f)
                            : sns_interp64<STRIDE>(scf, b + n2);
    else s = sns_interp64<STRIDE>(scf, b);
    return exp2_raw_fm(s);
}

// Side record for the synthesis kernel; a good frame makes the slot just written the stream's current one.
__device__ __forceinline__ void write_side(const EntropyParams& p, int srow, bool ok, int ltpf_active, int pitch_index,
                                           int nbits, int slot, int new_slot) {
    int32_t* sd = p.side + (size_t)srow * SIDE_WORDS;
    sd[SD_OK] = ok;
    sd[SD_LTPF_ACTIVE] = ok ? ltpf_active : 0;
    sd[SD_PITCH_INDEX] = ok ? pitch_index : 0;
    sd[SD_NBITS] = nbits;
    sd[SD_SLOT] = ok ? new_slot : slot;
    if (ok && p.fixed_slot < 0) p.sstate[(size_t)srow * SS_WORDS + SS_SLOT] = new_slot;
}

// ---------------------------------------------------------------- kernel 1b: integers -> shaped spectrum
// Dequantisation, residual refinement, noise filling, global gain, TNS lattice, SNS gains (reference D4-D8); one
// thread per frame, every thread walks all ne lines, so the warp stays converged without any work sorting.
template <int W /* noise-filling half width: 3 at 10 ms, 2 at 7.5 ms */, bool IDS>
__device__ __forceinline__ void dequant_body(const EntropyParams& p, const int block) {
    extern __shared__ __align__(16) uint8_t smem[];
    float* s_scf = (float*)smem;
    int32_t* s_band = (int32_t*)(s_scf + 16 * ENT_THREADS);
    uint8_t* s_rows = (uint8_t*)(s_band + 68);

    const DevConfig& c = *p.cfg;
    const int tid = threadIdx.x, lane = tid & 31;
    const int stream0 = block * ENT_THREADS;
    const int ne = c.ne;

    // hand-off record of this thread slot
    const int32_t* ho = p.handoff + (size_t)(stream0 + tid) * HO_WORDS;
    const int fid = ho[HO_FID];
    const int stream = stream0 + fid;
    const bool live = stream < p.n_streams;
    const int srow = live ? state_row<IDS>(p.ids, stream) : stream;   // the stream's persistent rows
    const bool ok = ho[HO_OK] != 0;
    SideInfoD si;
    si.lastnz = ho[HO_LASTNZ]; si.lsb_mode = ho[HO_LSB_MODE]; si.gg_ind = ho[HO_GG_IND]; si.bw = ho[HO_BW];
    si.num_tns = ho[HO_NUM_TNS]; si.noise_factor = ho[HO_NOISE_FACTOR];
    si.ind_lf = ho[HO_IND_LF]; si.ind_hf = ho[HO_IND_HF]; si.submode_msb = ho[HO_SUBMODE_MSB]; si.submode_lsb = ho[HO_SUBMODE_LSB];
    si.g_ind = ho[HO_G_IND]; si.ls_inda = ho[HO_LS_INDA]; si.ls_indb = ho[HO_LS_INDB]; si.idx_a = ho[HO_IDX_A]; si.idx_b = ho[HO_IDX_B];
    si.ltpf_active = ho[HO_LTPF_ACTIVE]; si.pitch_index = ho[HO_PITCH_INDEX];
    si.rc_in0 = si.rc_in1 = si.pitch_present = 0;
    const int rc_order0 = ho[HO_RC_ORDER0], rc_order1 = ho[HO_RC_ORDER1];
    const int nres = ho[HO_NRES];
    const uint32_t seed_acc = (uint32_t)ho[HO_SEED];
    int rc_i[16];
#pragma unroll
    for (int i = 0; i < 16; i++) rc_i[i] = ho[HO_RC_I + i];
    Reader rd;
    rd.buf = s_rows + fid * p.row_pitch;
    rd.len = ho[HO_LEN];
    rd.head = ho[HO_HEAD];
    rd.tail = ho[HO_TAIL];
    const int nbits = rd.len * 8;
    int32_t* xq = p.xq + ((size_t)((stream0 + tid) >> 5) * ne) * 32 + lane * 4;   // thread-private slice, line k at xq[xq_off(k)]

    for (int i = tid; i < 65; i += ENT_THREADS) s_band[i] = p.cfg->band_idx[i];
    // the frame bytes are only needed again for the residual bits (non-lsb mode); stage them when any frame of the CTA has some
    const bool need_rows = ok && !si.lsb_mode && nres > 0;
    if (__syncthreads_or(need_rows)) {
        stage_rows(p, s_rows, stream0, tid);
    }
    __syncthreads();
    {   // resume the tail reader mid-byte: (tail + tw_n) % 8 == 0
        const int idx = rd.len - 1 - (rd.tail >> 3);
        const uint32_t byte = (need_rows && idx >= 0 && idx < rd.len) ? rd.buf[idx] : 0u;
        rd.tw = (uint64_t)(byte >> (rd.tail & 7));
        rd.tw_n = 8 - (rd.tail & 7);
    }

    // ---- pass 2: dequantise, noise fill, gain, TNS, SNS; spectrum -> inactive slot
    int slot = 0;
    if (live && p.fixed_slot < 0) slot = p.sstate[(size_t)srow * SS_WORDS + SS_SLOT];
    const int new_slot = p.fixed_slot >= 0 ? p.fixed_slot : slot ^ 1;
    float* s_y = s_scf + tid;                                          // PVQ vector / scale factors, stride T
    bool is_zero_frame = false;
    FrameScalars fs{};
    TnsPlan tf{};
    int lastnz = 0;
    if (ok) {
        lastnz = si.lastnz;
        const int x0 = xq[0], x1 = xq[1];
        is_zero_frame = si.lastnz == 2 && x0 == 0 && x1 == 0 && si.gg_ind == 0;
        fs = frame_scalars(c, nbits, si.gg_ind, si.noise_factor, si.bw);
        tns_plan(tf, c, si.bw, si.num_tns, rc_order0, rc_order1, rc_i);
        // SNS: stage 1 + PVQ shape + DCT rotation -> 16 scale factors in s_y, evaluated per band on demand below
        const int shape_j = (si.submode_msb << 1) + si.submode_lsb;
        const float* gains;
        constexpr int YS = ENT_THREADS;
        switch (shape_j) {                                             // spectral_noise_shaping.rs:21-60
            case 0: {
                mpvq_deenum(10, 10, si.ls_inda, (uint32_t)si.idx_a, s_y, YS);
                // second call writes z[0..6) which the reference copies to y[10..16)
                mpvq_deenum(6, 1, si.ls_indb, (uint32_t)si.idx_b, s_y + 10 * YS, YS);
                gains = LC3T_SNS_VQ_REG_ADJ_GAINS;
                break;
            }
            case 1:
                mpvq_deenum(10, 10, si.ls_inda, (uint32_t)si.idx_a, s_y, YS);
                for (int i = 10; i < 16; i++) s_y[i * YS] = 0.0f;
                gains = LC3T_SNS_VQ_REG_LF_ADJ_GAINS;
                break;
            case 2: mpvq_deenum(16, 8, si.ls_inda, (uint32_t)si.idx_a, s_y, YS); gains = LC3T_SNS_VQ_NEAR_ADJ_GAINS; break;
            default: mpvq_deenum(16, 6, si.ls_inda, (uint32_t)si.idx_a, s_y, YS); gains = LC3T_SNS_VQ_FAR_ADJ_GAINS; break;
        }
        float y[16];
        const float g = sns_norm_gain(s_y, ENT_THREADS, gains, si.g_ind, y);
        for (int n = 0; n < 16; n++) s_y[n * ENT_THREADS] = sns_scale_factor(y, g, n, si.ind_lf, si.ind_hf);
    }
    const int nb = c.nb;

    // rows of one warp belong to arbitrary streams of the CTA (work sorting) and may sit in different slots
    // (a slot only flips on a good frame): every row is addressed through its own stream id and slot
    const size_t slot_stride = (size_t)p.slot_streams * ne;
    const long long my_row_off_ll = (long long)((size_t)new_slot * slot_stride + (size_t)srow * ne);

    const bool any_ok = __any_sync(0xffffffffu, ok);
    if (any_ok) {
        float st[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        float rc[8] = {0, 0, 0, 0, 0, 0, 0, 0};  // coefficient set in use
        int ord = 0, om = 0;                     // this lane's order in use, the warp's largest
        int tns_phase = 0, tns_next = ok ? tf.s0 : 0x7fffffff;    // next line at which this lane switches filters
        int last_nz = -1000;
        int nf_state = (int)(seed_acc & 0xffffu);
        int res_used = 0;
        // The integers come back four lines at a time (one 16-byte load per thread and group), three groups ahead of the
        // group in use, so the L2 round trip never sits on the serial per-line chain.  The line loop is unrolled over a
        // group: every lane walks the same line k, so k & 3 is static, a line and its look-ahead partner (k + W, for the
        // noise-filling window) are fixed registers of the group in use and the next one, and four finished lines leave
        // as one 16-byte store.  Groups beyond the frame's lastnz (even) are not fetched; their lines read as zero.
        const int n_valid = ok ? lastnz : 0;
        const int4* xg = (const int4*)xq;                              // group of lines b .. b + 3 of this thread at xg[(b / 4) * 32]
        auto fetch_group = [&](int b) -> int4 {                        // the load only: its result is not touched here
            int4 r = make_int4(0, 0, 0, 0);
            if (b < n_valid) r = xg[(b >> 2) * 32];
            return r;
        };
        auto trim_group = [&](int4 r, int b) -> int4 {                 // lines at and beyond lastnz hold stale integers
            if (b + 2 >= n_valid) { r.z = 0; r.w = 0; }
            return r;
        };
        int4 g = trim_group(fetch_group(0), 0), gn = trim_group(fetch_group(4), 4);
        int4 gnn = fetch_group(8);
        {
            const int32_t e[4] = {g.x, g.y, g.z, g.w};
#pragma unroll
            for (int j = 0; j < W; j++)
                if (e[j] != 0 && j < fs.bw_stop) last_nz = j;
        }
        const bool res_on = ok && !si.lsb_mode;
        const bool nf_on = ok && !is_zero_frame;
        // The four lines of group k4.  SW: some lane changes its TNS filter inside the group, so the switch is tested at
        // every line and the lattice runs at the warp's largest order of that line; otherwise at the compile-time depth OM.
        auto lines = [&](auto swc, auto omc, const int32_t (&e)[8], const float (&gl)[4], const int k4, float (&o)[4]) {
            constexpr bool SW = decltype(swc)::value;
            constexpr int OM = decltype(omc)::value;
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const int k = k4 + u;
                last_nz = (e[u + W] != 0 && k + W < fs.bw_stop) ? k + W : last_nz;
                const int32_t xi = e[u];
                float v = (float)xi;
                {   // one tail bit per non-zero line while the budget lasts (it cannot run past the frame here, see
                    // DESIGN.md); read straight from the staged row, no window to refill
                    const bool take = res_on && xi != 0 && res_used < nres;
                    const int bidx = max(rd.len - 1 - (rd.tail >> 3), 0);
                    const uint32_t bit = ((uint32_t)rd.buf[bidx] >> (rd.tail & 7)) & 1u;
                    v = take ? residual_refine(v, xi, bit) : v;
                    rd.tail += take ? 1 : 0;
                    res_used += take ? 1 : 0;
                }
                v = noise_fill(nf_on && k >= fs.nf_start && k < fs.bw_stop && last_nz < k - W, nf_state, fs.nf_level, v);
                v = xm(v, fs.gg);
                if constexpr (SW) {
                    if (k == tns_next) tns_switch(tf, rc, ord, tns_phase, tns_next);
                    om = __reduce_max_sync(0xffffffffu, ord);
                }
                v = tns_lattice_line(v, rc, st, ord, SW ? om : OM);
                o[u] = ok ? xm(v, gl[u]) : v;
            }
        };
        // lines are walked band by band: the bands that start inside a group are entered (warp-uniformly) before its
        // lines, each line then uses the gain of its own band
        int band = -1, k_end = 0;
        float gband = 0.0f;
        float4* outp = (float4*)(p.spec + my_row_off_ll);
        for (int k4 = 0; k4 < ne; k4 += 4) {
            const int4 g3 = fetch_group(k4 + 12);                       // three groups ahead; first touched a group later
            float gl[4] = {gband, gband, gband, gband};
            while (k_end < k4 + 4) {
                band++;
                gband = ok ? sns_band_gain<ENT_THREADS>(s_y, band, nb) : 0.0f;
                const int first = k_end - k4;
                k_end = band + 1 < nb ? s_band[band + 1] : ne;
#pragma unroll
                for (int u = 0; u < 4; u++) gl[u] = u >= first ? gband : gl[u];
            }
            const int32_t e[8] = {g.x, g.y, g.z, g.w, gn.x, gn.y, gn.z, gn.w};
            const bool any_sw = __any_sync(0xffffffffu, (unsigned)(tns_next - k4) < 4u);
            float o[4];
            if (!any_sw) {
                // No lane changes its TNS filter inside this group (all but two or three groups of a frame): the four
                // lines are ONE basic block - selects only, the lattice at a compile-time depth that covers the warp's
                // largest order - so the scheduler overlaps the lines' chains: stage j of a line needs the state stage
                // j - 1 of the previous line left, i.e. consecutive lines run two lattice stages apart, not eight.
                if (om == 0) lines(std::false_type{}, std::integral_constant<int, 0>{}, e, gl, k4, o);
                else if (om <= 4) lines(std::false_type{}, std::integral_constant<int, 4>{}, e, gl, k4, o);
                else lines(std::false_type{}, std::integral_constant<int, 8>{}, e, gl, k4, o);
            } else {
                lines(std::true_type{}, std::integral_constant<int, 8>{}, e, gl, k4, o);
            }
            // four finished lines leave as one 16-byte store into the thread's own stream-major row (the two halves of
            // a 32-byte sector are written four lines apart and meet in L2)
            if (ok) *outp = make_float4(o[0], o[1], o[2], o[3]);
            outp++;
            g = gn;
            gn = trim_group(gnn, k4 + 8);
            gnn = g3;
        }
    }

    if (live) write_side(p, srow, ok, si.ltpf_active, si.pitch_index, nbits, slot, new_slot);
}

// 5 CTAs per SM (96 registers): measured against 4 (119 registers, 0.80 ms), 6 (80, 0.74 ms) and 7 (72, spills, 0.82 ms): 0.667 ms
template <int W, bool IDS>
__global__ void __launch_bounds__(ENT_THREADS, 5) dequant_kernel(const __grid_constant__ EntropyParams p) {
    dequant_body<W, IDS>(p, blockIdx.x);
}

template <int W>
__global__ void __launch_bounds__(ENT_THREADS, 5) dequant_mixed_kernel(const __grid_constant__ MixedParams m) {
    __shared__ EntropyParams s_p;
    __shared__ int s_block;
    mixed_select(m, &s_p, &s_block, 1);
    dequant_body<W, false>(s_p, s_block);
}

// ---------------------------------------------------------------- kernels 1b' / 1b'': the small-batch dequantisation
// The thread-per-frame dequant_kernel needs ~100 k frames to fill the GPU: every frame's ne lines are one thread's serial
// loop (0.07 ms at 16 384 streams of 120 lines whatever the occupancy).  Up to DQW_MAX_STREAMS streams the same work is
// split along what is really serial:
//   dequant_warp_kernel (one WARP per frame, a lane owns the lines k = lane, lane + 32, ...): everything but the lattice.
//     * residual refinement and noise filling are per-line decisions whose only serial part is a COUNT (the i-th
//       non-zero line takes the i-th residual bit; the i-th filled line takes the LCG's i-th output): ballot + popcount
//       give the rank, and the LCG is jumped to any rank with the composed multiplier / increment table
//       DevConfig::nf_lcg;
//     * the noise-filling window test (no non-zero integer within +-W lines) is a mask test on the ballots of three rows;
//     * SNS scale factors: PVQ de-enumeration on one lane, the 16 x 16 rotation on 16 lanes, band gains on 64;
//     * frames without TNS leave finished; a frame with an active TNS filter leaves its gain-scaled lines and its 64
//       band gains, and appends itself to a list;
//   tns_list_kernel (one THREAD per listed frame): the TNS lattice - a true recurrence over lines - then the SNS gains,
//     in place on the frame's spectrum row, with the select-based lattice so the warp never splits.
// The three kernels share one definition of each reference step (above dequant_body), so the f32 operations per line are
// the same in the same order: the spectrum is bit-identical (tested).
constexpr int DQW_WARPS = 8;
__host__ __device__ inline size_t dequant_warp_smem_bytes() {
    return sizeof(float) * DQW_WARPS * (64 + 16 + 16) + MAX_NE;
}

template <bool IDS>
__device__ __forceinline__ void dequant_warp_body(const EntropyParams& p, const int block) {
    extern __shared__ __align__(16) uint8_t smem[];
    float* s_gband = (float*)smem;                                     // [DQW_WARPS][64]
    float* s_scf = s_gband + DQW_WARPS * 64;                           // [DQW_WARPS][16]
    float* s_y = s_scf + DQW_WARPS * 16;                               // [DQW_WARPS][16]
    uint8_t* s_band_of = (uint8_t*)(s_y + DQW_WARPS * 16);             // line -> band

    const DevConfig& c = *p.cfg;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int ne = c.ne, nb = c.nb;
    const int W = c.n_ms == LC3B_10MS ? 3 : 2;
    const uint32_t lt_mask = (1u << lane) - 1u;

    for (int k = tid; k < ne; k += DQW_WARPS * 32) {                   // the last band runs to ne
        int lo = 0, hi = nb - 1;
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (c.band_idx[mid] <= k) lo = mid; else hi = mid - 1;
        }
        s_band_of[k] = (uint8_t)lo;
    }
    __syncthreads();                                                   // the only CTA-wide step: warps are independent below

    // ---- hand-off record of this warp's thread slot (the entropy kernel's tid)
    const int n_slots = ((p.n_streams + ENT_THREADS - 1) / ENT_THREADS) * ENT_THREADS;
    const int slot = block * DQW_WARPS + wid;
    if (slot >= n_slots) return;
    const int32_t* ho = p.handoff + (size_t)slot * HO_WORDS;
    const int h0 = ho[lane];
    const int h1 = lane < HO_WORDS - 32 ? ho[32 + lane] : 0;
    // both shuffles are executed by every lane whatever i is (a lane-dependent i must not split the warp around them)
    auto field = [&](int i) -> int {
        const int a = __shfl_sync(0xffffffffu, h0, i & 31), b = __shfl_sync(0xffffffffu, h1, i & 31);
        return i < 32 ? a : b;
    };
    const int fid = field(HO_FID);
    const int stream = (slot / ENT_THREADS) * ENT_THREADS + fid;
    const bool live = stream < p.n_streams;
    const int srow = live ? state_row<IDS>(p.ids, stream) : stream;   // the stream's persistent rows
    const bool ok = live && field(HO_OK) != 0;
    const int lastnz = field(HO_LASTNZ), lsb_mode = field(HO_LSB_MODE), gg_ind = field(HO_GG_IND), bw = field(HO_BW);
    const int num_tns = field(HO_NUM_TNS), noise_factor = field(HO_NOISE_FACTOR);
    const int rc_order0 = field(HO_RC_ORDER0), rc_order1 = field(HO_RC_ORDER1);
    const int nres = field(HO_NRES), tail = field(HO_TAIL), len = field(HO_LEN);
    const uint32_t seed0 = (uint32_t)field(HO_SEED) & 0xffffu;
    const int ltpf_active = field(HO_LTPF_ACTIVE), pitch_index = field(HO_PITCH_INDEX);
    const int nbits = len * 8;

    int slot_cur = 0;
    if (live && p.fixed_slot < 0) slot_cur = p.sstate[(size_t)srow * SS_WORDS + SS_SLOT];
    const int new_slot = p.fixed_slot >= 0 ? p.fixed_slot : slot_cur ^ 1;
    constexpr int NR = (MAX_NE + 31) / 32;                             // rows of 32 lines
    if (ok) {                                                          // warp-uniform
        const FrameScalars fs = frame_scalars(c, nbits, gg_ind, noise_factor, bw);
        // does any TNS filter of this frame do anything?  (phase 2 exists only for bw >= 3, temporal_noise_shaping.rs:83-138)
        const bool has_tns = rc_order0 > 0 || (bw >= 3 && num_tns == 2 && rc_order1 > 0);
        // ---- SNS scale factors -> 64 band gains
        float* scf = s_scf + wid * 16;
        float* yv = s_y + wid * 16;
        float* gband = s_gband + wid * 64;
        {
            const int ind_lf = field(HO_IND_LF), ind_hf = field(HO_IND_HF), submode_msb = field(HO_SUBMODE_MSB);
            const int submode_lsb = field(HO_SUBMODE_LSB), g_ind = field(HO_G_IND), ls_inda = field(HO_LS_INDA);
            const int ls_indb = field(HO_LS_INDB), idx_a = field(HO_IDX_A), idx_b = field(HO_IDX_B);
            const int shape_j = (submode_msb << 1) + submode_lsb;
            if (lane == 0) {                                            // the thread kernel's switch, see there
                switch (shape_j) {
                    case 0:
                        mpvq_deenum(10, 10, ls_inda, (uint32_t)idx_a, yv, 1);
                        mpvq_deenum(6, 1, ls_indb, (uint32_t)idx_b, yv + 10, 1);
                        break;
                    case 1:
                        mpvq_deenum(10, 10, ls_inda, (uint32_t)idx_a, yv, 1);
                        for (int i = 10; i < 16; i++) yv[i] = 0.0f;
                        break;
                    case 2: mpvq_deenum(16, 8, ls_inda, (uint32_t)idx_a, yv, 1); break;
                    default: mpvq_deenum(16, 6, ls_inda, (uint32_t)idx_a, yv, 1); break;
                }
            }
            __syncwarp();
            if (lane < 16) {
                const float* gains = shape_j == 0 ? LC3T_SNS_VQ_REG_ADJ_GAINS : shape_j == 1 ? LC3T_SNS_VQ_REG_LF_ADJ_GAINS
                                     : shape_j == 2 ? LC3T_SNS_VQ_NEAR_ADJ_GAINS : LC3T_SNS_VQ_FAR_ADJ_GAINS;
                float y[16];
                const float g = sns_norm_gain(yv, 1, gains, g_ind, y);
                scf[lane] = sns_scale_factor(y, g, lane, ind_lf, ind_hf);
            }
            __syncwarp();
            for (int b0 = 0; b0 < 64; b0 += 32) {
                const int b = b0 + lane;
                if (b < nb) gband[b] = sns_band_gain<1>(scf, b, nb);
            }
            __syncwarp();
        }
        // ---- integers of this frame: thread slot's lane-interleaved scratch column
        const int32_t* xq = p.xq + ((size_t)(slot >> 5) * ne) * 32 + (slot & 31) * 4;
        int32_t x[NR];
        uint32_t nzb[NR];                                              // non-zero lines below bw_stop, one bit per line
#pragma unroll
        for (int j = 0; j < NR; j++) {
            const int k = 32 * j + lane;
            x[j] = (32 * j < ne && k < lastnz) ? xq[xq_off(k)] : 0;    // lastnz <= ne
            nzb[j] = __ballot_sync(0xffffffffu, x[j] != 0 && k < fs.bw_stop);
        }
        const bool is_zero_frame = lastnz == 2 && (__ballot_sync(0xffffffffu, x[0] != 0) & 3u) == 0 && gg_ind == 0;
        const uint8_t* fr = p.frames + (size_t)stream * p.frame_stride;
        float* dst = p.spec + ((size_t)new_slot * p.slot_streams + srow) * ne;
        int res_base = 0, fill_base = 0;
#pragma unroll
        for (int j = 0; j < NR; j++) {
            if (32 * j < ne) {                                         // warp-uniform
                const int k = 32 * j + lane;
                const int32_t xi = x[j];
                float v = (float)xi;
                {   // residual_spectrum.rs:13-39: the i-th non-zero line takes the i-th tail bit while the budget lasts
                    const uint32_t m = __ballot_sync(0xffffffffu, xi != 0);
                    const int rank = res_base + __popc(m & lt_mask);
                    res_base += __popc(m);
                    const bool take = !lsb_mode && xi != 0 && rank < nres;
                    const int pos = tail + rank;
                    const int bidx = max(len - 1 - (pos >> 3), 0);
                    const uint32_t bit = take ? ((uint32_t)fr[bidx] >> (pos & 7)) & 1u : 0u;
                    v = take ? residual_refine(v, xi, bit) : v;
                }
                {   // noise_filling.rs:37-55: lines whose +-W neighbourhood holds no non-zero integer
                    const uint32_t lo = j > 0 ? nzb[j > 0 ? j - 1 : 0] : 0u, mid = nzb[j], hi = j + 1 < NR ? nzb[j + 1 < NR ? j + 1 : j] : 0u;
                    const uint64_t a = ((uint64_t)mid << 32) | lo, b = ((uint64_t)hi << 32) | mid;
                    const uint32_t wm = (1u << (W + 1)) - 1u;
                    const uint32_t near = ((uint32_t)(a >> (32 + lane - W)) | (uint32_t)(b >> lane)) & wm;
                    const bool fill = !is_zero_frame && k >= fs.nf_start && k < fs.bw_stop && near == 0;
                    const uint32_t fm = __ballot_sync(0xffffffffu, fill);
                    const int n = fill_base + __popc(fm & lt_mask) + 1;     // this line takes the LCG's n-th output
                    fill_base += __popc(fm);
                    const uint32_t ac = c.nf_lcg[fill ? n : 0];
                    const uint32_t st = ((ac >> 16) * seed0 + (ac & 0xffffu)) & 0xffffu;
                    v = fill ? nf_fill_level(st, fs.nf_level) : v;
                }
                v = xm(v, fs.gg);
                if (k < ne) dst[k] = has_tns ? v : xm(v, gband[s_band_of[k]]);   // coalesced row
            }
        }
        if (has_tns) {                                                 // the lattice kernel finishes this frame
            float* gb = p.gband + (size_t)slot * 64;
            gb[lane] = lane < nb ? gband[lane] : 0.0f;
            gb[32 + lane] = 32 + lane < nb ? gband[32 + lane] : 0.0f;
            if (lane == 0) p.tns_list[2 + atomicAdd(p.tns_list, 1)] = slot;
        }
    }
    if (live && lane == 0) write_side(p, srow, ok, ltpf_active, pitch_index, nbits, slot_cur, new_slot);
}

// The listed frames' lattices, one thread each: temporal_noise_shaping.rs:24-74 then the SNS gains, four lines at a time
// in place on the frame's row (the row is the slot dequant_warp_kernel just wrote and made current).
template <bool IDS>
__device__ __forceinline__ void tns_list_body(const EntropyParams& p, const int block) {
    // band gains of the CTA's frames, [band][thread] (a thread walks its own column: no bank conflicts), and the band edges:
    // the walk along the bands must not wait for global memory at every band change
    __shared__ float s_g[64 * ENT_THREADS];
    __shared__ int s_edge[65];
    const DevConfig& c = *p.cfg;
    const int tid = (int)threadIdx.x;
    const int i = block * ENT_THREADS + tid;
    // tns_list = [count, CTAs done, thread slots ...].  Every CTA reads the count first and reports when it is through; the
    // last one to report empties the list for the next call (no kernel of the next call can be running yet).
    const int count = p.tns_list[0];
    const int n_ctas = (p.n_streams + ENT_THREADS - 1) / ENT_THREADS;
    auto report_done = [&]() {
        __syncthreads();
        if (tid == 0 && atomicAdd(p.tns_list + 1, 1) == n_ctas - 1) { p.tns_list[0] = 0; p.tns_list[1] = 0; }
    };
    if (block * ENT_THREADS >= count) { report_done(); return; }       // whole CTA beyond the list
    const bool mine = i < count;
    const int slot = mine ? p.tns_list[2 + i] : 0;
    const int32_t* ho = p.handoff + (size_t)slot * HO_WORDS;
    const int ne = c.ne, nb = c.nb;
    for (int b = tid; b < 65; b += ENT_THREADS) s_edge[b] = b < nb ? c.band_idx[b] : 0x7fffffff;   // the last band runs to ne
    if (mine) {
        const float4* gb4 = (const float4*)(p.gband + (size_t)slot * 64);
#pragma unroll
        for (int q = 0; q < 16; q++) {
            const float4 g4 = gb4[q];
            s_g[(4 * q + 0) * ENT_THREADS + tid] = g4.x;
            s_g[(4 * q + 1) * ENT_THREADS + tid] = g4.y;
            s_g[(4 * q + 2) * ENT_THREADS + tid] = g4.z;
            s_g[(4 * q + 3) * ENT_THREADS + tid] = g4.w;
        }
    }
    TnsPlan tf{};
    float* row = p.spec;
    if (mine) {
        const int stream = state_row<IDS>(p.ids, (slot / ENT_THREADS) * ENT_THREADS + ho[HO_FID]);   // listed frames are live
        tns_plan(tf, c, ho[HO_BW], ho[HO_NUM_TNS], ho[HO_RC_ORDER0], ho[HO_RC_ORDER1], ho + HO_RC_I);
        const int cur = p.fixed_slot >= 0 ? p.fixed_slot : p.sstate[(size_t)stream * SS_WORDS + SS_SLOT];
        row = p.spec + ((size_t)cur * p.slot_streams + stream) * ne;
    }
    __syncthreads();
    float st[8] = {0, 0, 0, 0, 0, 0, 0, 0}, rc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    int ord = 0, om = 0, phase = 0, next = mine ? tf.s0 : 0x7fffffff;
    int band = 0, band_end = mine ? s_edge[1] : 0x7fffffff;
    float gcur = mine ? s_g[tid] : 0.0f;
    const int n4 = ne >> 2;                                            // ne is a multiple of 4 in every configuration
    const float4 zero4 = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    float4 cur4 = mine ? ((const float4*)row)[0] : zero4;
    float4 nxt4 = (mine && 1 < n4) ? ((const float4*)row)[1] : zero4;
    for (int g = 0; g < n4; g++) {
        const float4 nn4 = (mine && g + 2 < n4) ? ((const float4*)row)[g + 2] : zero4;     // two groups ahead of the lattice
        float vv[4] = {cur4.x, cur4.y, cur4.z, cur4.w};
#pragma unroll
        for (int e = 0; e < 4; e++) {
            const int k = 4 * g + e;
            float v = vv[e];
            const bool sw = k == next;
            if (__any_sync(0xffffffffu, sw)) {
                if (sw) tns_switch(tf, rc, ord, phase, next);
                om = __reduce_max_sync(0xffffffffu, ord);
            }
            v = tns_lattice_line(v, rc, st, ord, om);
            while (k >= band_end) {                                    // next band; zero-width bands are skipped
                band++;
                band_end = s_edge[band + 1 < 64 ? band + 1 : 64];
                gcur = s_g[band * ENT_THREADS + tid];
            }
            vv[e] = xm(v, gcur);
        }
        if (mine) ((float4*)row)[g] = make_float4(vv[0], vv[1], vv[2], vv[3]);
        cur4 = nxt4;
        nxt4 = nn4;
    }
    report_done();
}

template <bool IDS>
__global__ void __launch_bounds__(DQW_WARPS * 32) dequant_warp_kernel(const __grid_constant__ EntropyParams p) {
    dequant_warp_body<IDS>(p, blockIdx.x);
}
template <bool IDS>
__global__ void __launch_bounds__(ENT_THREADS) tns_list_kernel(const __grid_constant__ EntropyParams p) {
    tns_list_body<IDS>(p, blockIdx.x);
}

// mixed-rate variants
__global__ void __launch_bounds__(DQW_WARPS * 32) dequant_warp_mixed_kernel(const __grid_constant__ MixedParams m) {
    __shared__ EntropyParams s_p;
    __shared__ int s_block;
    mixed_select(m, &s_p, &s_block, ENT_THREADS / DQW_WARPS);
    dequant_warp_body<false>(s_p, s_block);
}
__global__ void __launch_bounds__(ENT_THREADS) tns_list_mixed_kernel(const __grid_constant__ MixedParams m) {
    __shared__ EntropyParams s_p;
    __shared__ int s_block;
    mixed_select(m, &s_p, &s_block, 1);
    tns_list_body<false>(s_p, s_block);
}

int entropy_row_pitch(int nbytes) {
    int words = (nbytes + 3) / 4 + 1;
    if ((words & 1) == 0) words++;                 // odd word pitch: lanes land on distinct banks
    return words * 4;
}

// dynamic shared memory limits, once per handle (lc3b_decoder_init) for the largest frame the handle accepts
cudaError_t prepare_entropy(const DecoderState& st) {
    const int pitch = entropy_row_pitch(st.max_nbytes);
    const int es = (int)entropy_smem_bytes(pitch), ds = (int)dequant_smem_bytes(pitch);
    cudaError_t e = cudaFuncSetAttribute(entropy_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, es);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(entropy_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, es);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(entropy_mixed_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, es);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(dequant_kernel<3, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, ds);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(dequant_kernel<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, ds);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(dequant_kernel<3, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, ds);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(dequant_kernel<2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, ds);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(dequant_mixed_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, ds);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(dequant_mixed_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, ds);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(dequant_warp_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dequant_warp_smem_bytes());
    if (e == cudaSuccess) e = cudaFuncSetAttribute(dequant_warp_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dequant_warp_smem_bytes());
    if (e == cudaSuccess) e = cudaFuncSetAttribute(dequant_warp_mixed_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dequant_warp_smem_bytes());
    return e;
}

EntropyParams entropy_params(const DecoderState& st, const uint8_t* frames, const int32_t* frame_nbytes, int nbytes,
                             size_t frame_stride, int32_t* status_out, int base, int count, const int32_t* ids) {
    EntropyParams p;
    memset(&p, 0, sizeof(p));                      // padding bytes are part of the graph cache key
    // a sub-batch is the same launch with every per-stream pointer moved to its first stream (base is a multiple of the
    // CTA's 128 thread slots, so the lane-interleaved scratch moves by whole blocks); only the stride between the two
    // spectrum slots still belongs to the whole handle.  A subset call's rows reach the state through the id list:
    // only the row-indexed pointers and the id list move, the state pointers (sb) stay at the handle's first stream.
    const size_t b = (size_t)base, sb = ids ? 0 : b;
    const int ne = st.cfg.ne;
    p.cfg = st.dcfg;
    p.frames = frames ? frames + b * frame_stride : nullptr;
    p.frame_nbytes = frame_nbytes ? frame_nbytes + b : nullptr;
    p.nbytes = nbytes;
    p.frame_stride = frame_stride;
    p.n_streams = count < 0 ? st.n_streams : count;
    p.slot_streams = st.n_streams;
    p.spec = st.spec + sb * ne;
    p.xq = st.xq + b * ne;                         // [block32][ne][32]: 32 streams are ne * 32 integers
    p.handoff = st.handoff + b * HO_WORDS;
    p.side = st.side + sb * SIDE_WORDS;
    p.sstate = st.sstate + sb * SS_WORDS;
    p.status_out = status_out ? status_out + b : nullptr;
    p.trace = st.trace ? st.trace + b * LC3B_TRACE_WORDS : nullptr;
    p.trace_x = st.trace_x ? st.trace_x + b * ne : nullptr;
    p.sym_lut = st.sym_lut;
    p.gband = st.gband;                            // small-batch path only (never split)
    p.tns_list = st.tns_list;
    p.nsym_prev = st.nsym_prev ? st.nsym_prev + sb : nullptr;
    p.fixed_slot = st.fixed_slot;
    p.min_nbytes = st.min_nbytes;
    p.row_pitch = entropy_row_pitch(nbytes);
    p.ids = ids ? ids + b : nullptr;
    return p;
}

// n_call: rows of the whole call (not of this sub-batch): the small-batch kernels share one list per handle, so the choice
// between them and dequant_kernel is made once per call
template <bool IDS>
static void plan_entropy_kernels(LaunchPlan& plan, const DecoderState& st, const EntropyParams& p, int stages, int first_dep, int n_call) {
    const unsigned grid = (unsigned)((p.n_streams + ENT_THREADS - 1) / ENT_THREADS);
    int dep = first_dep;
    if (stages & 1) { plan.add(entropy_kernel<IDS>, grid, ENT_THREADS, entropy_smem_bytes(p.row_pitch), p, dep); dep = -2; }
    if (stages & 2) {
        if (use_dequant_warp(n_call, st.dequant_mode)) {               // never split (its list is per handle)
            plan.add(dequant_warp_kernel<IDS>, grid * (ENT_THREADS / DQW_WARPS), DQW_WARPS * 32, dequant_warp_smem_bytes(), p, dep);
            plan.add(tns_list_kernel<IDS>, grid, ENT_THREADS, 0, p);
        } else {
            const size_t smem = dequant_smem_bytes(p.row_pitch);
            if (st.cfg.n_ms == LC3B_10MS) plan.add(dequant_kernel<3, IDS>, grid, ENT_THREADS, smem, p, dep);
            else plan.add(dequant_kernel<2, IDS>, grid, ENT_THREADS, smem, p, dep);
        }
    }
}

// stages: bit 0 entropy_kernel (bitstream -> integers), bit 1 dequant_kernel (integers -> shaped spectrum)
void plan_entropy(LaunchPlan& plan, const DecoderState& st, const uint8_t* frames, const int32_t* frame_nbytes, int nbytes,
                  size_t frame_stride, int32_t* status_out, int stages, int base, int count, int first_dep,
                  const int32_t* ids, int n_rows) {
    const EntropyParams p = entropy_params(st, frames, frame_nbytes, nbytes, frame_stride, status_out, base, count, ids);
    if (ids) plan_entropy_kernels<true>(plan, st, p, stages, first_dep, n_rows);
    else plan_entropy_kernels<false>(plan, st, p, stages, first_dep, st.n_streams);
}

// Which dequantisation kernel a batch of n streams gets: warp-per-frame below DQW_MAX_STREAMS (it finishes a small batch
// in a fraction of the thread-per-frame kernel's serial latency but costs more issue slots per frame), thread-per-frame
// above.  lc3b_decoder_set_dequant_mode (or LC3B_DEQUANT=warp|thread in the environment) forces one; tests run both.
constexpr int DQW_MAX_STREAMS = 12288;        // measured cross-over at 16 kHz / 7.5 ms: 12-16 k streams (profiles/r2_small_batch.json)
bool use_dequant_warp(int n_streams, int mode) {
    static const int forced = [] {
        const char* e = getenv("LC3B_DEQUANT");
        return !e ? 0 : (e[0] == 'w' ? 1 : e[0] == 't' ? 2 : 0);
    }();
    if (mode == 0) mode = forced;
    if (mode) return mode == 1;
    return n_streams <= DQW_MAX_STREAMS;
}

// From this many streams (or units of a time-parallel call) a decode call is issued as four independent sub-batches
// (run_decode in lc3b_api.cu): measured at 48 kHz / 150 B, 65 536 streams gain 7 %, 131 072 18 %, 262 144 10 %, 32 768 nothing.
int decode_split_min_streams() { return 65536; }

// Mixed-rate call: one entropy launch over all buckets, one dequantisation launch per frame duration present.
// Returns the node index of the 10 ms and of the 7.5 ms dequantisation launch (-1 if absent) for the synthesis nodes
// to depend on.
void plan_entropy_mixed(LaunchPlan& plan, const MixedTables& t, const uint8_t* frames, const int32_t* frame_nbytes, int nbytes,
                        size_t frame_stride, int32_t* status_out, int* node_d10, int* node_d75) {
    MixedParams m;
    memset(&m, 0, sizeof(m));
    m.frames = frames;
    m.frame_nbytes = frame_nbytes;
    m.nbytes = nbytes;
    m.frame_stride = frame_stride;
    m.status_out = status_out;
    m.row_pitch = entropy_row_pitch(nbytes);
    m.buckets = t.all;
    m.n_buckets = t.n_all;
    const int e = plan.add(entropy_mixed_kernel, (unsigned)t.cta_all, ENT_THREADS, entropy_smem_bytes(m.row_pitch), m, -1);
    const size_t smem = dequant_smem_bytes(m.row_pitch);
    *node_d10 = *node_d75 = -1;
    if (use_dequant_warp(t.n_streams, t.dequant_mode)) {               // one launch for both frame durations (W is a run-time value there)
        const int a = plan.add(dequant_warp_mixed_kernel, (unsigned)(t.cta_all * (ENT_THREADS / DQW_WARPS)), DQW_WARPS * 32,
                               dequant_warp_smem_bytes(), m, e);
        *node_d10 = *node_d75 = plan.add(tns_list_mixed_kernel, (unsigned)t.cta_all, ENT_THREADS, 0, m, a);
        return;
    }
    if (t.n_10 > 0) {
        m.buckets = t.b10;
        m.n_buckets = t.n_10;
        *node_d10 = plan.add(dequant_mixed_kernel<3>, (unsigned)t.cta_10, ENT_THREADS, smem, m, e);
    }
    if (t.n_75 > 0) {
        m.buckets = t.b75;
        m.n_buckets = t.n_75;
        *node_d75 = plan.add(dequant_mixed_kernel<2>, (unsigned)t.cta_75, ENT_THREADS, smem, m, e);
    }
}

}  // namespace lc3b
