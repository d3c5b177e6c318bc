// File-level callers of the hot path, after the reference's examples (SURVEY.md 8f-2), on the C++ host mirror:
//   lc3b_codec_file encode in.wav out.lc3 <fs> <ms> <nbytes_per_channel>     examples/encode.rs:37-116
//   lc3b_codec_file decode in.lc3 out.wav <fs> <ms> <nbytes_per_channel> <channels>   examples/decode.rs:37-123
//   lc3b_codec_file wavtest                                                  wav.rs:130-148 (no GPU needed)
// Channels of the file are the streams of one batched handle; each direction runs time-parallel calls over many frame
// periods (lc3b_encode_stream_frames / lc3b_decode_stream_frames) instead of one call per period.
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <iterator>
#include <string>
#include <vector>

#include "../include/lc3b.hpp"
#include "../include/lc3b_file.hpp"

using namespace lc3b;

static std::vector<uint8_t> slurp(const char* path) {
    std::ifstream f(path, std::ios::binary);
    if (!f) { std::fprintf(stderr, "cannot open %s\n", path); std::exit(2); }
    return std::vector<uint8_t>((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
}
static SamplingFrequency fs_of(int hz) {
    switch (hz) {
        case 8000: return SamplingFrequency::Hz8000;
        case 16000: return SamplingFrequency::Hz16000;
        case 24000: return SamplingFrequency::Hz24000;
        case 32000: return SamplingFrequency::Hz32000;
        case 44100: return SamplingFrequency::Hz44100;
        case 48000: return SamplingFrequency::Hz48000;
    }
    std::fprintf(stderr, "unsupported sampling frequency %d\n", hz);
    std::exit(2);
}
static FrameDuration dur_of(const std::string& ms) { return ms == "7.5" ? FrameDuration::SevenPointFiveMs : FrameDuration::TenMs; }
#define CUDA_OK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { std::fprintf(stderr, "%s: %s\n", #x, cudaGetErrorString(e_)); std::exit(3); } } while (0)

static int wavtest() {
    const uint8_t buffer[] = {0x52, 0x49, 0x46, 0x46, 0x16, 0x29, 0x0B, 0x00, 0x57, 0x41, 0x56, 0x45, 0x66, 0x6D, 0x74, 0x20, 0x10, 0x00,
                              0x00, 0x00, 0x01, 0x00, 0x02, 0x00, 0x44, 0xAC, 0x00, 0x00, 0x10, 0xB1, 0x02, 0x00, 0x04, 0x00, 0x10, 0x00,
                              0x64, 0x61, 0x74, 0x61, 0x70, 0x28, 0x0B, 0x00, 0x00};
    wav::WavHeader h;
    if (wav::read_header(buffer, sizeof(buffer), &h)) return 1;
    if (h.num_channels != 2 || h.sample_rate != 44100 || h.byte_rate != 176400 || h.block_align != 4 || h.bits_per_sample != 16 ||
        h.data_size != 731248 || h.data_start_position != 44)
        return 1;
    uint8_t out[44];
    size_t n = 0;
    if (wav::write_header(h, out, sizeof(out), &n) || n != 44) return 1;
    for (int i = 0; i < 44; i++) if (out[i] != buffer[i]) return 1;
    if (!wav::write_header(h, out, 10, &n)) return 1;                    // WriteHeaderBufferTooSmall
    if (wav::read_header(buffer, 20, &h) != wav::WavError::ReadHeaderInvalidHeaderLength) return 1;
    std::puts("wavtest ok");
    return 0;
}

static int encode(const char* wav_name, const char* lc3_name, int hz, const std::string& ms, size_t nbytes) {
    const std::vector<uint8_t> in = slurp(wav_name);
    wav::WavHeader wh;
    if (auto e = wav::read_header(in.data(), in.size(), &wh)) { std::fprintf(stderr, "wav error %d\n", (int)*e); return 2; }
    const size_t nch = wh.num_channels;
    const SamplingFrequency f = fs_of(hz);
    const FrameDuration d = dur_of(ms);
    const size_t ws_bytes = Lc3BatchEncoder::calc_working_buffer_lengths(nch, d, f, nbytes);
    void* ws = nullptr;
    CUDA_OK(cudaMalloc(&ws, ws_bytes));
    Lc3BatchEncoder enc(nch, d, f, ws, ws_bytes, nbytes);
    const size_t nf = (size_t)enc.config.nf, bytes_per_frame = nf * nch * 2;
    const size_t data_bytes = in.size() > wh.data_start_position ? in.size() - wh.data_start_position : 0;
    const size_t periods = (data_bytes + bytes_per_frame - 1) / bytes_per_frame;               // encode.rs:73
    // up to CHUNK frame periods per time-parallel call, staged channel-major: [nch][F][nf] in, [nch][F][nbytes] out
    constexpr size_t CHUNK = 4096;
    const size_t max_f = std::min(periods, CHUNK);
    std::vector<int16_t> period(nch * nf), staged(nch * max_f * nf);
    std::vector<uint8_t> bits(nch * max_f * nbytes);
    int16_t* d_pcm = nullptr;
    uint8_t* d_bits = nullptr;
    void* d_scratch = nullptr;
    const size_t scratch_bytes = max_f ? enc.multi_scratch_bytes(max_f) : 0;
    if (max_f) {
        CUDA_OK(cudaMalloc((void**)&d_pcm, staged.size() * sizeof(int16_t)));
        CUDA_OK(cudaMalloc((void**)&d_bits, bits.size()));
        CUDA_OK(cudaMalloc(&d_scratch, scratch_bytes));
    }
    std::ofstream out(lc3_name, std::ios::binary);
    for (size_t p0 = 0; p0 < periods; p0 += CHUNK) {
        const size_t F = std::min(CHUNK, periods - p0);
        for (size_t p = 0; p < F; p++) {
            const size_t cur = wh.data_start_position + (p0 + p) * bytes_per_frame;
            const size_t avail = std::min(in.size() - cur, bytes_per_frame) / (2 * nch);
            deinterleave(in.data() + cur, avail, nf, nch, period.data());
            for (size_t c = 0; c < nch; c++) std::memcpy(staged.data() + (c * F + p) * nf, period.data() + c * nf, nf * sizeof(int16_t));
        }
        CUDA_OK(cudaMemcpy(d_pcm, staged.data(), nch * F * nf * sizeof(int16_t), cudaMemcpyHostToDevice));
        enc.encode_stream_frames(d_pcm, F, d_bits, nbytes, nbytes, d_scratch, scratch_bytes);
        CUDA_OK(cudaMemcpy(bits.data(), d_bits, nch * F * nbytes, cudaMemcpyDeviceToHost));
        for (size_t p = 0; p < F; p++)
            for (size_t c = 0; c < nch; c++) out.write((const char*)bits.data() + (c * F + p) * nbytes, (std::streamsize)nbytes);
    }
    std::printf("encoded %zu frame periods x %zu channels in %zu calls\n", periods, nch, (periods + CHUNK - 1) / CHUNK);
    cudaFree(d_pcm); cudaFree(d_bits); cudaFree(d_scratch); cudaFree(ws);
    return 0;
}

static int decode(const char* lc3_name, const char* wav_name, int hz, const std::string& ms, size_t nbytes, size_t nch) {
    const std::vector<uint8_t> in = slurp(lc3_name);
    const SamplingFrequency f = fs_of(hz);
    const FrameDuration d = dur_of(ms);
    const size_t ws_bytes = Lc3BatchDecoder::calc_working_buffer_lengths(nch, d, f, nbytes);
    void* ws = nullptr;
    CUDA_OK(cudaMalloc(&ws, ws_bytes));
    Lc3BatchDecoder dec(nch, d, f, ws, ws_bytes, nbytes);
    const size_t nf = (size_t)dec.config.nf;
    const Lc3File lf{nch, nbytes};
    const size_t periods = lf.frame_periods(in.size());
    // the whole file in ONE time-parallel call (SURVEY.md 8f-1): channel-major staging [nch][periods][nbytes]
    std::vector<uint8_t> staged(nch * periods * nbytes);
    for (size_t p = 0; p < periods; p++)
        for (size_t c = 0; c < nch; c++)
            std::memcpy(staged.data() + (c * periods + p) * nbytes, lf.channel_frame(in.data(), p, c), nbytes);
    uint8_t* d_frames = nullptr;
    int16_t* d_pcm = nullptr;
    void* d_scratch = nullptr;
    const size_t scratch_bytes = periods ? dec.multi_scratch_bytes(periods) : 0;
    std::vector<int16_t> by_channel(nch * periods * nf);
    std::vector<uint8_t> pcm(periods * nf * nch * 2);
    if (periods) {
        CUDA_OK(cudaMalloc((void**)&d_frames, staged.size()));
        CUDA_OK(cudaMalloc((void**)&d_pcm, by_channel.size() * sizeof(int16_t)));
        CUDA_OK(cudaMalloc(&d_scratch, scratch_bytes));
        CUDA_OK(cudaMemcpy(d_frames, staged.data(), staged.size(), cudaMemcpyHostToDevice));
        if (dec.decode_stream_frames(16, d_frames, nbytes, periods, d_pcm, d_scratch, scratch_bytes)) {
            std::fprintf(stderr, "decoder error\n");
            return 2;
        }
        CUDA_OK(cudaMemcpy(by_channel.data(), d_pcm, by_channel.size() * sizeof(int16_t), cudaMemcpyDeviceToHost));
        std::vector<int16_t> period(nch * nf);
        for (size_t p = 0; p < periods; p++) {
            for (size_t c = 0; c < nch; c++) std::memcpy(period.data() + c * nf, by_channel.data() + (c * periods + p) * nf, nf * sizeof(int16_t));
            interleave(period.data(), nf, nch, pcm.data() + p * nf * nch * 2);
        }
        cudaFree(d_frames); cudaFree(d_pcm); cudaFree(d_scratch);
    }
    wav::WavHeader wh;
    wh.num_channels = nch;
    wh.sample_rate = (size_t)dec.config.fs;
    wh.bits_per_sample = 16;
    wh.block_align = nch * 2;
    wh.byte_rate = wh.sample_rate * wh.block_align;
    wh.data_size = pcm.size();                                            // (the reference's example leaves the sizes at 0)
    wh.data_start_position = wav::FULL_WAV_HEADER_LEN;
    wh.data_with_header_size = pcm.size() + wav::FULL_WAV_HEADER_LEN - wav::RIFF_HEADER_ONLY_LEN;
    uint8_t hdr[wav::FULL_WAV_HEADER_LEN];
    wav::write_header(wh, hdr, sizeof(hdr), nullptr);
    std::ofstream out(wav_name, std::ios::binary);
    out.write((const char*)hdr, sizeof(hdr));
    out.write((const char*)pcm.data(), (std::streamsize)pcm.size());
    std::printf("decoded %zu frame periods x %zu channels in one call\n", periods, nch);
    cudaFree(ws);
    return 0;
}

int main(int argc, char** argv) {
    const std::string mode = argc > 1 ? argv[1] : "";
    try {
        if (mode == "wavtest") return wavtest();
        if (mode == "encode" && argc == 7) return encode(argv[2], argv[3], std::atoi(argv[4]), argv[5], (size_t)std::atoi(argv[6]));
        if (mode == "decode" && argc == 8)
            return decode(argv[2], argv[3], std::atoi(argv[4]), argv[5], (size_t)std::atoi(argv[6]), (size_t)std::atoi(argv[7]));
    } catch (const std::exception& e) {
        std::fprintf(stderr, "%s\n", e.what());
        return 4;
    }
    std::fprintf(stderr, "usage: %s encode in.wav out.lc3 fs ms nbytes | decode in.lc3 out.wav fs ms nbytes channels | wavtest\n", argv[0]);
    return 2;
}
