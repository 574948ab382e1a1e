// projectultra_b200/csrc/pu_internal.h — shared internals of libpu_b200.so (not part of the C ABI).
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <complex>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <functional>
#include <string>
#include <type_traits>
#include <vector>

#include "pu/pu_capi.h"

namespace pu {

void set_error(const char* fmt, ...);

#define PU_CUDA_TRY(expr)                                                                       \
    do {                                                                                        \
        cudaError_t _e = (expr);                                                                \
        if (_e != cudaSuccess) {                                                                \
            ::pu::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return PU_ERR_CUDA;                                                                 \
        }                                                                                       \
    } while (0)

#define PU_REQUIRE(cond, msg)                     \
    do {                                          \
        if (!(cond)) {                            \
            ::pu::set_error("%s", msg);           \
            return PU_ERR_INVALID;                \
        }                                         \
    } while (0)

// Grow-only device / pinned-host scratch buffer.
struct Buffer {
    void* ptr = nullptr;
    size_t cap = 0;
    bool pinned_host = false;
    pu_status reserve(size_t bytes);
    void release();
};

// Device copy of a host table, owned by a handle and freed with it.
struct DevMem {
    void* p = nullptr;
    DevMem() = default;
    DevMem(const DevMem&) = delete;
    DevMem& operator=(const DevMem&) = delete;
    ~DevMem() { if (p) cudaFree(p); }
    template <class T>
    pu_status upload(const T* src, size_t n) {
        if (p) { cudaFree(p); p = nullptr; }
        PU_CUDA_TRY(cudaMalloc(&p, n * sizeof(T) > 16 ? n * sizeof(T) : 16));
        if (n) {
            // A pageable H2D cudaMemcpy may return once the source is staged, before the DMA has landed, and the kernels that
            // read these tables run on NON-BLOCKING streams (no implicit ordering with the legacy stream): wait for it.
            PU_CUDA_TRY(cudaMemcpy(p, src, n * sizeof(T), cudaMemcpyHostToDevice));
            PU_CUDA_TRY(cudaStreamSynchronize(cudaStreamLegacy));
        }
        return PU_OK;
    }
};

// The PU_MEM_HOST side of a batch entry point: the call declares its host arrays, each with the device pointer its body reads,
// then run() moves the batch through the context's pinned and device staging buffers in slabs of whole rows.  Per slab: one packed
// H2D copy, the body on device pointers (the entry point's PU_MEM_DEVICE path on `st`), one packed D2H copy, a synchronise of `st`.
// Every staged array starts on a 256-byte boundary (the TMA paths check sample addresses); a NULL host array stays NULL.
class HostStage {
public:
    HostStage(pu_ctx* ctx, cudaStream_t st, size_t B) : ctx_(ctx), st_(st), B_(B) {}
    // per-row arrays: `row` elements of row b are read from / written to host + b * host_stride and packed on the device
    template <class T> void in(const T** dev, const T* host, size_t row, size_t host_stride = 0) { add(kIn, dev, host, row, host_stride); }
    // output rows come back as the body left them, zero-filled before it runs
    template <class T> void out(T** dev, T* host, size_t row, size_t host_stride = 0) { add(kOut, dev, host, row, host_stride); }
    // the caller's bytes go down and come back: in-place rows, or rows the body writes only in part
    template <class T> void inout(T** dev, T* host, size_t row, size_t host_stride = 0) { add(kInOut, dev, host, row, host_stride); }
    // one array of n elements for the whole call
    template <class T> void whole(const T** dev, const T* host, size_t n) { add(kWhole, dev, host, n, n); }
    // body(nb) runs on nb rows at the declared device pointers; B == 0 runs nothing
    pu_status run(const std::function<pu_status(size_t nb)>& body);

private:
    enum Kind { kWhole, kIn, kInOut, kOut };   // the order of the staged layout: H2D covers [whole, inout], D2H [inout, out]
    struct Array {
        Kind kind;
        std::function<void(void*)> bind;
        char* host;
        size_t row, stride, off;   // bytes
    };
    template <class P, class T>
    void add(Kind k, P** dev, T* host, size_t row, size_t host_stride) {
        arrays_.push_back({k, [dev](void* d) { *dev = static_cast<P*>(d); }, reinterpret_cast<char*>(const_cast<std::remove_const_t<T>*>(host)),
                           row * sizeof(T), (host_stride ? host_stride : row) * sizeof(T), 0});
    }
    pu_ctx* ctx_;
    cudaStream_t st_;
    size_t B_;
    std::vector<Array> arrays_;
};

}  // namespace pu

namespace pu {
// One lane of the host-buffer pipeline (pu_receive_decode_batch with PU_MEM_HOST): its own stream and buffers, so
// that the H2D copy of slab i+1 overlaps the kernels and the D2H copy of slab i.
struct PipeSlot {
    cudaStream_t stream = nullptr;
    Buffer d_in, d_llr, d_out, h_in, h_out;
    size_t off = 0, nb = 0;   // slab in flight (nb == 0: idle)
};
}  // namespace pu

struct pu_ctx {
    int device = 0;
    int sm_count = 0;
    int cc_major = 0, cc_minor = 0;
    cudaStream_t stream = nullptr;  // context-owned stream used when the caller passes NULL
    std::atomic<uint64_t> launches{0};
    std::atomic<uint64_t> h2d_bytes{0}, d2h_bytes{0};   // bytes moved by the host-buffer pipeline (pu_receive_decode_batch, PU_MEM_HOST)
    pu::Buffer stage_dev, stage_host;                   // pu::HostStage: staging of PU_MEM_HOST calls
    pu::Buffer d_aux;                                   // LLR scratch of pu_receive_decode_batch
    pu::Buffer f_bytes, f_ok, f_iters;                  // scratch of pu_frame_decode_batch (grow-only, reused across calls)
    pu::PipeSlot pipe[2];
    cudaEvent_t pipe_ev = nullptr;
    // scratch of pu_linksim_run (sweep.cu), grow-only and reused across calls: [0..6] batch buffers (rx, llr, info, ok, iters, n_llr, sync),
    // [7 + 4 s .. 10 + 4 s] slot s = {pinned descriptors, device descriptors, device counters, pinned counters},
    // [15..17] fresh payloads {TX rows, payload rows, noise levels}, [18..19] frame modes {reassembled frames, frame_len + info + ncw},
    // [20] coded bytes of fresh payloads (pu_linksim_run_raw)
    pu::Buffer cfo_mix;            // pu_channel_apply_cfo_batch: (cos, sin)(2 pi 1500 i / fs) per sample index, host libm
    size_t cfo_mix_len = 0;
    uint32_t cfo_mix_fs = 0;
    pu::Buffer sweep[21];
    cudaEvent_t sweep_ev[2] = {nullptr, nullptr};
};

namespace pu {
// PU_MEM_DEVICE: `stream` is the caller's stream, NULL meaning the CUDA default stream (as in the runtime API);
// PU_MEM_HOST: NULL selects the context's own non-blocking stream for the staged copies and the kernel.
inline cudaStream_t pick_stream(pu_ctx* ctx, void* stream, pu_memspace space = PU_MEM_HOST) {
    if (stream || space == PU_MEM_DEVICE) return reinterpret_cast<cudaStream_t>(stream);
    return ctx->stream;
}
}  // namespace pu

// chirp_sync.cu: dual-chirp synchronisation shared by the OFDM_CHIRP and MC-DPSK receive entry points
namespace pu {
struct ChirpDev {
    int n, gap;                        // chirp samples (24 000), gap samples (4 800)
    float fs, cfo_to_samples;          // sample rate; sample_rate / chirp_rate
    const float* up_s; const float* up_c; const float* dn_s; const float* dn_c;   // templates (generateTemplate, chirp_sync.hpp:706-735)
    float up_e, dn_e;                  // template energies
    // ranking pass of the two-tier coarse search (chirp_sync.cu): the templates taken every 6th sample and scaled by 6,
    // {up sin, up cos, down sin, down cos} x nd floats, and the 47-tap low-pass in front of the 6:1 decimation of the samples
    const float* dec; const float* lp; int nd;
};
// templates of the 300 -> 2700 Hz, 500 ms chirp pair with 100 ms gaps (OFDMChirpWaveform::getChirpConfig, ofdm_chirp_waveform.cpp:39-49 ==
// MultiCarrierDPSKConfig::getChirpConfig, multi_carrier_dpsk.hpp:78-88): host table of 4 n floats {up sin, up cos, down sin, down cos}
// followed by the ranking tables (4 nd decimated template floats, 64 low-pass taps);
// the caller uploads it and chirp_dev_bind points the descriptor at the device copy
void chirp_templates_host(float fs, std::vector<float>& table, ChirpDev& c);
inline void chirp_dev_bind(ChirpDev& c, const float* dev_table) {
    c.up_s = dev_table; c.up_c = dev_table + c.n; c.dn_s = dev_table + 2 * static_cast<size_t>(c.n); c.dn_c = dev_table + 3 * static_cast<size_t>(c.n);
    c.dec = dev_table + 4 * static_cast<size_t>(c.n);
    c.lp = c.dec + 4 * static_cast<size_t>(c.nd);
}
void tools_apply_cfo(float* samples, size_t n, float cfo_hz, float sample_rate);     // tools_cfo.cpp
// tables of tools_apply_cfo: tw[fft_size / 2] twiddles exp(-2 pi i k / fft_size) from the float angle, rot[n] = (cos, sin) of the float
// phase recurrence; the device injector (tools_cfo_gpu.cu) uploads the same tables
void tools_cfo_twiddles(size_t fft_size, std::complex<float>* tw);
void tools_cfo_rotator(size_t n, float cfo_hz, float sample_rate, std::complex<float>* rot);
// frame_v2.cu: the body of pu_frame_decode_batch, enqueue only, on caller-owned device scratch: llr[B][num_codewords][648] ->
// cw_bytes[B * num_codewords][k / 8], cw_ok, cw_iters -> frame_out[B][frame_cap], frame_len[B], info[B][5].  ncw_per[b] (NULL = all
// num_codewords) is the number of codewords frame b delivered, as RxPipeline::decodeFrame's num_codewords.
pu_status frame_decode_enqueue(pu_ctx* ctx, pu_ldpc* dec, const float* llr, size_t B, int num_codewords, const int32_t* ncw_per,
                               uint8_t* cw_bytes, uint8_t* cw_ok, int32_t* cw_iters, uint8_t* frame_out, size_t frame_cap, int32_t* frame_len,
                               int32_t* info, cudaStream_t st);
// linksim.cu: whole-frame counters (linksim.FRAME_COUNTER_NAMES) of frames decoded by frame_decode_enqueue against the frames sent
// (row tx_index[b] of sent[][sent_stride], sent_len bytes each, n_cw codewords): counters[bin[b]][6] += {1, lost, info[3], n_cw,
// info[4] == 0, 0}
pu_status count_frame_errors(pu_ctx* ctx, const uint8_t* frame_out, size_t frame_cap, const int32_t* frame_len, const int32_t* info,
                             const uint8_t* sent, size_t sent_stride, const uint32_t* tx_index, const uint32_t* bin, size_t sent_len, int n_cw,
                             size_t B, uint64_t* counters, cudaStream_t st);
// linksim.cu: the body of pu_count_raw_errors on the caller's stream (pre-decoder counters {soft_bits, erasures, bit_errors, strong_errors}).
// il_step != 0: the rows were deinterleaved by ChannelInterleaver(step = il_step, 648) codeword by codeword after the receiver wrote them,
// and n_valid[b] counts soft bits in the receiver's (delivered) order, so the erasures past it are found through the permutation.
pu_status count_raw_errors(pu_ctx* ctx, const float* llr, size_t llr_stride, size_t n_bits, const int32_t* n_valid, const uint8_t* coded,
                           size_t coded_stride, const uint32_t* coded_index, const uint32_t* bin, size_t B, float strong, uint64_t* counters,
                           cudaStream_t st, uint32_t il_step = 0);
// ldpc_decode.cu: ChannelInterleaver(bits_per_symbol, 648) of pu_channel_interleaver_perm, perm[i] = i * step mod 648.  The inverse of
// step mod 648 (transmitted bit j of a codeword is coded bit j * step^-1 mod 648), and ChannelInterleaver::interleave of n_cw packed
// 81-byte codewords in place, each on its own.
uint32_t channel_interleaver_inverse_step(size_t bits_per_symbol);
void channel_interleave_codewords(size_t bits_per_symbol, uint8_t* coded, size_t n_cw);
// interleave.cu: the body of pu_llr_deinterleave_batch on device pointers, enqueue only
pu_status llr_deinterleave_enqueue(pu_ctx* ctx, float* llr, size_t B, size_t llr_stride, size_t n_blocks, size_t bits_per_symbol, cudaStream_t st);
float channel_power_sum(const float* tx, size_t L);                                   // channel.cu: the two halves of pu_channel_noise_std
float channel_noise_std_from_sum(float acc, size_t L, float snr_db, int convention);
cudaError_t chirp_search_stats(unsigned long long* out);
cudaError_t chirp_phase_cycles(unsigned long long* out);   // [8] thread-0 cycles per phase of the two-tier search, then cleared   // {searches, rounds} since the last call, then cleared
cudaError_t chirp_detect_launch(const ChirpDev& c, const float* samples, size_t B, size_t frame_stride, int L, float threshold, int sym_len,
                                int4* out_info, float4* out_f, int* frame_start, int* frame_nsym, float* cfo_out, float* phase_out,
                                int* n_llr, int llr_per_symbol, int llr_stride, cudaStream_t st);
}  // namespace pu
