// lc3b engine: the opaque handle types of the C ABI (include/lc3b.h), shared by the translation units that implement it.
#pragma once
#include <vector>

#include "lc3b_common.cuh"
#include "lc3b_plan.cuh"

namespace lc3b {
// The host-side id list of a subset call (lc3b_decode_frames_subset and friends): every id in [0, n_streams) and none
// listed twice.  A stream is marked with the call's epoch, so a check is O(n) and the marks are never cleared (except
// when the epoch wraps).  The accepted list is kept in `ids`, a pageable copy: cudaMemcpyAsync has consumed a pageable
// source by the time it returns, so the caller's array is only read during the call even when it is pinned.
struct IdList {
    std::vector<uint32_t> mark;
    std::vector<int32_t> ids;
    uint32_t epoch = 0;
    bool take(const int32_t* in, int n, int n_streams) {
        if ((int)mark.size() != n_streams) mark.assign((size_t)n_streams, 0u);
        if (++epoch == 0) { mark.assign((size_t)n_streams, 0u); epoch = 1; }
        ids.resize((size_t)n);
        for (int i = 0; i < n; i++) {
            const int32_t s = in[i];
            if (s < 0 || s >= n_streams || mark[(size_t)s] == epoch) return false;
            mark[(size_t)s] = epoch;
            ids[(size_t)i] = s;
        }
        return true;
    }
};

// The host-side plan of a ragged time-parallel call (lc3b_decode_stream_frames_subset, lc3b_encode_stream_frames_subset):
// an id list as for a subset call and a frame count per row.  Row i's frames are the call's units off_i .. off_i + count_i - 1,
// off_i the exclusive prefix sum of the counts in the caller's order.  The rows with frames become the row table
// (lc3b_common.cuh), sorted by count, descending, with a stable LSD radix sort: one pass per byte of the largest count,
// so planning is O(n_rows) and never touches a unit.  Like IdList the table is a pageable copy that one cudaMemcpyAsync
// sends to the front of the caller's scratch.
struct RowTable {
    std::vector<int32_t> words, tmp;
    long long total = 0;
    int n_live = 0;                       // rows with frames = rows of the table
    // false for a bad or duplicate id, a negative count or more than max_total frames in all
    bool take(IdList& idl, const int32_t* ids, const int32_t* counts, int n_rows, int n_streams, long long max_total) {
        if (n_rows < 0 || n_rows > n_streams || !idl.take(ids, n_rows, n_streams)) return false;
        words.resize((size_t)n_rows * RT_WORDS);
        tmp.resize(words.size());
        total = 0;
        n_live = 0;
        int32_t cmax = 0;
        for (int i = 0; i < n_rows; i++) {
            const int32_t c = counts[i];
            if (c < 0 || total + c > max_total) return false;
            if (c > 0) {
                int32_t* w = &words[(size_t)n_live++ * RT_WORDS];
                w[RT_ROW] = idl.ids[(size_t)i];
                w[RT_OFF] = (int32_t)total;
                w[RT_COUNT] = c;
                if (c > cmax) cmax = c;
            }
            total += c;
        }
        for (int shift = 0; shift < 32 && (cmax >> shift) != 0; shift += 8) {
            size_t start[257] = {0};
            auto digit = [&](int r) { return 255 - ((words[(size_t)r * RT_WORDS + RT_COUNT] >> shift) & 255); };
            for (int r = 0; r < n_live; r++) start[digit(r) + 1]++;
            for (int d = 0; d < 256; d++) start[d + 1] += start[d];
            for (int r = 0; r < n_live; r++) {
                const size_t dst = start[digit(r)]++;
                for (int k = 0; k < RT_WORDS; k++) tmp[dst * RT_WORDS + k] = words[(size_t)r * RT_WORDS + k];
            }
            words.swap(tmp);
        }
        return true;
    }
    cudaError_t send(void* scratch, cudaStream_t stream) const {
        return cudaMemcpyAsync(scratch, words.data(), sizeof(int32_t) * RT_WORDS * (size_t)n_live, cudaMemcpyHostToDevice, stream);
    }
};
}  // namespace lc3b

struct lc3b_decoder {
    lc3b::DecoderState st{};
    int stage_mask = 7;
    // how a call's kernels are issued: 0 = one launch each on the caller's stream, 1 = one cached CUDA graph per call
    int graph_mode = 0;
    lc3b::GraphCache graphs;
    // a large batch is issued as up to four independent sub-batches on auxiliary streams (run_decode in lc3b_api.cu)
    int split = 0;                        // 0 = by batch size, 1 = never, 2 / 4 = that many sub-batches
    lc3b::PlanLanes lanes;
    // optional pipelining of the host entry point: PCM leaves on an internal copy stream from a double-buffered
    // staging area, so the device->host copy of call i overlaps the kernels of call i+1
    int pipelined = 0;
    int buf = 0;
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t compute_done[2] = {nullptr, nullptr}, d2h_done[2] = {nullptr, nullptr};
    bool d2h_pending[2] = {false, false};
    lc3b::IdList id_list;                 // subset calls and resets (lc3b_decode_frames_subset, lc3b_decoder_reset_streams)
    lc3b::RowTable row_table;             // ragged time-parallel calls (lc3b_decode_stream_frames_subset)
};

namespace lc3b {

// one thread-local slot for the last CUDA error of any entry point (decoder, encoder, mixed, sharded)
int cuda_fail(cudaError_t e);
#define LC3B_CU(x)                                         \
    do {                                                   \
        cudaError_t _e = (x);                              \
        if (_e != cudaSuccess) return lc3b::cuda_fail(_e); \
    } while (0)

// graph mode default: LC3B_GRAPH=0/1 in the environment overrides; otherwise graphs are used for batches small enough
// to be launch-sensitive
int default_graph_mode(int n_streams);

// internals of lc3b_api.cu used by the mixed-rate and sharded front ends
bool config_new(int sampling_frequency, int frame_duration, lc3b_config* c);
int decoder_workspace_bytes(int n_streams, int frame_duration, int sampling_frequency, int max_nbytes, bool staging,
                            size_t* device_bytes);
int decoder_init(lc3b_decoder** out, int n_streams, int frame_duration, int sampling_frequency, int max_nbytes, int device,
                 void* dev_workspace, size_t workspace_bytes, void* cuda_stream, bool staging);

// Restores the caller's current CUDA device when it goes out of scope (the init functions select the handle's device).
struct DeviceGuard {
    int prev = -1;
    DeviceGuard() { if (cudaGetDevice(&prev) != cudaSuccess) prev = -1; }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

}  // namespace lc3b
