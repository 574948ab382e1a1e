// projectultra_b200/csrc/linksim.cu — the batched Monte-Carlo link: (channel ->) demodulate -> LDPC decode ->
// count frame / bit errors, chained on one stream with all intermediates resident in HBM.
//
// Reference behaviour: the trial loop of the reference's Monte-Carlo tools, e.g. tools/test_mode_snr.cpp:40-105 and
// tools/test_ofdm_chirp_pilots.cpp:166-260: per trial  channel.process -> demodulator.processPresynced ->
// getSoftBits (first 648) -> LDPCDecoder::decodeSoft -> success iff lastDecodeSuccess() AND decoded bytes == payload
// (test_mode_snr.cpp:98-104).  Trials are independent, so here they are the batch dimension.
#include <algorithm>
#include <memory>
#include <new>

#include <cstdlib>

#include "pu_internal.h"

// implemented in ofdm_demod.cu / ldpc_decode.cu
extern "C" pu_status pu_ofdm_presynced_batch(pu_ofdm*, const float*, size_t, size_t, int, const float*, const float*,
                                             float*, size_t, float*, float*, pu_memspace, void*);
extern "C" pu_status pu_ldpc_decode_batch(pu_ldpc*, const float*, size_t, size_t, uint8_t*, size_t, uint8_t*, int32_t*,
                                          pu_memspace, void*);
extern "C" int pu_ldpc_info_bits(const pu_ldpc*);
extern "C" int pu_ofdm_symbol_samples(const pu_ofdm*);
extern "C" int pu_ofdm_bits_per_symbol(const pu_ofdm*);
pu_ctx* pu_ofdm_context(pu_ofdm* h);   // ofdm_demod.cu
bool pu_ofdm_diff512_window(pu_ofdm* h, const float* d_samples, size_t B, size_t L, int training, int* first, int* n_symbols, int* sym_len,
                            int* cp, int* nfft);   // ofdm_demod.cu

namespace pu {

// counters[bin][6] = {frames, frame_errors, bit_errors, bits, decode_failures, iteration_sum}
// Bins below kSharedBins are accumulated in a per-CTA shared-memory table first (a sweep has tens of SNR points and
// neighbouring frames belong to different points), so global memory sees one atomic per (CTA, bin, counter) instead of
// five per frame on a few dozen addresses.
constexpr int kSharedBins = 64;
__global__ void __launch_bounds__(1024) count_errors_kernel(const uint8_t* __restrict__ info, size_t info_stride, const uint8_t* __restrict__ ok,
                                    const int32_t* __restrict__ iters, const uint8_t* __restrict__ payload_pool,
                                    size_t payload_stride, const uint32_t* __restrict__ tx_index,
                                    const uint32_t* __restrict__ bin, int payload_bytes, size_t B,
                                    unsigned long long* __restrict__ counters) {
    __shared__ unsigned long long local[kSharedBins * 6];
    for (int i = threadIdx.x; i < kSharedBins * 6; i += blockDim.x) local[i] = 0ull;
    __syncthreads();
    const size_t b = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
    if (b < B) {
        const uint8_t* got = info + b * info_stride;
        const uint8_t* want = payload_pool + static_cast<size_t>(tx_index ? tx_index[b] : 0) * payload_stride;
        int bit_err = 0;
        for (int i = 0; i < payload_bytes; ++i) bit_err += __popc(static_cast<unsigned>(got[i] ^ want[i]));
        const int decoded = ok[b] != 0;
        const int success = decoded && bit_err == 0;   // tools/test_mode_snr.cpp:98-104
        const size_t bi = bin ? bin[b] : 0;
        unsigned long long* c = bi < kSharedBins ? local + bi * 6 : counters + bi * 6;
        atomicAdd(&c[0], 1ull);
        if (!success) atomicAdd(&c[1], 1ull);
        if (bit_err) atomicAdd(&c[2], static_cast<unsigned long long>(bit_err));
        atomicAdd(&c[3], static_cast<unsigned long long>(payload_bytes) * 8ull);
        if (!decoded) atomicAdd(&c[4], 1ull);
        atomicAdd(&c[5], static_cast<unsigned long long>(iters ? iters[b] : 0));
    }
    __syncthreads();
    for (int i = threadIdx.x; i < kSharedBins * 6; i += blockDim.x)
        if (local[i]) atomicAdd(&counters[i], local[i]);
}

// Whole-frame rule (linksim.FrameLinkSim): a trial succeeds iff decodeFrame succeeded, the reassembled frame has the length of the frame
// sent and the same bytes.  One warp per frame; counters[bin][6] = {frames, frame_errors, codewords_failed, codewords, header_failures, 0}.
__global__ void __launch_bounds__(256) count_frame_errors_kernel(const uint8_t* __restrict__ frame_out, size_t frame_cap,
                                                                 const int32_t* __restrict__ frame_len, const int32_t* __restrict__ info,
                                                                 const uint8_t* __restrict__ sent, size_t sent_stride,
                                                                 const uint32_t* __restrict__ tx_index, const uint32_t* __restrict__ bin,
                                                                 int sent_len, int n_cw, size_t B, unsigned long long* __restrict__ counters) {
    const int lane = threadIdx.x & 31;
    const size_t b = blockIdx.x * static_cast<size_t>(blockDim.x >> 5) + (threadIdx.x >> 5);
    if (b >= B) return;
    const int32_t* in = info + b * 5;
    bool good = in[0] == 1 && frame_len[b] == sent_len;
    if (good) {
        const uint8_t* got = frame_out + b * frame_cap;
        const uint8_t* want = sent + static_cast<size_t>(tx_index ? tx_index[b] : 0) * sent_stride;
        bool same = true;
        for (int i = lane; i < sent_len; i += 32) same &= got[i] == want[i];
        good = __all_sync(0xffffffffu, same);
    }
    if (lane != 0) return;
    unsigned long long* c = counters + static_cast<size_t>(bin ? bin[b] : 0) * 6;
    atomicAdd(&c[0], 1ull);
    if (!good) atomicAdd(&c[1], 1ull);
    if (in[3]) atomicAdd(&c[2], static_cast<unsigned long long>(in[3]));
    atomicAdd(&c[3], static_cast<unsigned long long>(n_cw));
    if (in[4] == 0) atomicAdd(&c[4], 1ull);
}

pu_status count_frame_errors(pu_ctx* ctx, const uint8_t* frame_out, size_t frame_cap, const int32_t* frame_len, const int32_t* info,
                             const uint8_t* sent, size_t sent_stride, const uint32_t* tx_index, const uint32_t* bin, size_t sent_len, int n_cw,
                             size_t B, uint64_t* counters, cudaStream_t st) {
    PU_REQUIRE(sent_len <= frame_cap && sent_len <= sent_stride, "count_frame_errors: frame longer than its buffers");
    if (B == 0) return PU_OK;
    (void)cudaGetLastError();
    count_frame_errors_kernel<<<static_cast<unsigned>((B + 7) / 8), 256, 0, st>>>(frame_out, frame_cap, frame_len, info, sent, sent_stride, tx_index,
                                                                                 bin, static_cast<int>(sent_len), n_cw, B,
                                                                                 reinterpret_cast<unsigned long long*>(counters));
    ctx->launches.fetch_add(1);
    PU_CUDA_TRY(cudaGetLastError());
    return PU_OK;
}

// Pre-decoder counters (pu_count_raw_errors): counters[bin][4] = {soft_bits, erasures, bit_errors, strong_errors}.  Each warp takes a
// contiguous range of rows; neighbouring rows of a sweep batch share their bin (one work unit), so a lane keeps its counts in registers
// while the bin stays the same and the warp sums them into the global table only when it changes: a few atomics per (warp, unit) instead
// of per soft bit or per row.  Soft bits past n_valid are not read.  il_step != 0: the row was deinterleaved codeword by codeword with
// ChannelInterleaver(step = il_step, 648), so n_valid counts soft bits in DELIVERED order: decoder bit c * 648 + i came from delivered
// position c * 648 + (i * il_step mod 648), and it is an erasure when that position is >= n_valid.
__global__ void __launch_bounds__(256) count_raw_errors_kernel(const float* __restrict__ llr, size_t llr_stride, int n_bits, int il_step,
                                                               const int32_t* __restrict__ n_valid, const uint8_t* __restrict__ coded,
                                                               size_t coded_stride, const uint32_t* __restrict__ coded_index,
                                                               const uint32_t* __restrict__ bin, size_t B, size_t rows_per_warp, float strong,
                                                               unsigned long long* __restrict__ counters) {
    const int lane = threadIdx.x & 31;
    const size_t b0 = ((blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x) >> 5) * rows_per_warp;
    const size_t b1 = min(B, b0 + rows_per_warp);
    if (b0 >= b1) return;
    unsigned long long c[4] = {0ull, 0ull, 0ull, 0ull};
    uint32_t cur = bin ? bin[b0] : 0u;
    auto flush = [&]() {
        for (int i = 0; i < 4; ++i)
            for (int o = 16; o > 0; o >>= 1) c[i] += __shfl_xor_sync(0xffffffffu, c[i], o);
        if (lane == 0)
            for (int i = 0; i < 4; ++i)
                if (c[i]) atomicAdd(&counters[static_cast<size_t>(cur) * 4 + i], c[i]);
        c[0] = c[1] = c[2] = c[3] = 0ull;
    };
    for (size_t b = b0; b < b1; ++b) {
        const uint32_t bb = bin ? bin[b] : 0u;
        if (bb != cur) {
            flush();
            cur = bb;
        }
        const float* x = llr + b * llr_stride;
        const uint8_t* want = coded + static_cast<size_t>(coded_index ? coded_index[b] : b) * coded_stride;
        const int nv = n_valid ? min(max(n_valid[b], 0), n_bits) : n_bits;
        const bool permuted = il_step && nv < n_bits;
        if (lane == 0) {
            c[0] += static_cast<unsigned long long>(n_bits);
            if (!permuted) c[1] += static_cast<unsigned long long>(n_bits - nv);
        }
        for (int j = lane; j < (permuted ? n_bits : nv); j += 32) {
            if (permuted) {
                const int cw = j / PU_LDPC_N, i = j - cw * PU_LDPC_N;
                if (cw * PU_LDPC_N + i * il_step % PU_LDPC_N >= nv) { ++c[1]; continue; }
            }
            const float v = x[j];
            if (v == 0.0f) { ++c[1]; continue; }                      // +0 and -0
            const unsigned sent = (want[j >> 3] >> (7 - (j & 7))) & 1u;
            if ((v < 0.0f ? 1u : 0u) != sent) {
                ++c[2];
                if (fabsf(v) >= strong) ++c[3];
            }
        }
    }
    flush();
}

pu_status count_raw_errors(pu_ctx* ctx, const float* llr, size_t llr_stride, size_t n_bits, const int32_t* n_valid, const uint8_t* coded,
                           size_t coded_stride, const uint32_t* coded_index, const uint32_t* bin, size_t B, float strong, uint64_t* counters,
                           cudaStream_t st, uint32_t il_step) {
    PU_REQUIRE(n_bits <= llr_stride && (n_bits + 7) / 8 <= coded_stride && n_bits < (size_t(1) << 30),
               "pu_count_raw_errors: rows shorter than n_bits soft / coded bits");
    if (B == 0 || n_bits == 0) return PU_OK;
    const size_t warps = std::min<size_t>(B, static_cast<size_t>(std::max(ctx->sm_count, 1)) * 64);
    const size_t per = (B + warps - 1) / warps;
    const size_t blocks = ((B + per - 1) / per + 7) / 8;
    (void)cudaGetLastError();
    count_raw_errors_kernel<<<static_cast<unsigned>(blocks), 256, 0, st>>>(llr, llr_stride, static_cast<int>(n_bits), static_cast<int>(il_step), n_valid,
                                                                          coded, coded_stride,
                                                                          coded_index, bin, B, per, strong,
                                                                          reinterpret_cast<unsigned long long*>(counters));
    ctx->launches.fetch_add(1);
    PU_CUDA_TRY(cudaGetLastError());
    return PU_OK;
}

}  // namespace pu

extern "C" {

pu_status pu_count_raw_errors(pu_ctx* ctx, const float* llr, size_t llr_stride, size_t n_bits, const int32_t* n_valid, const uint8_t* coded,
                              size_t coded_stride, const uint32_t* coded_index, const uint32_t* bin, size_t B, float strong, uint64_t* counters,
                              void* stream) {
    PU_REQUIRE(ctx && counters && (B == 0 || (llr && coded)), "pu_count_raw_errors: NULL argument");
    PU_CUDA_TRY(cudaSetDevice(ctx->device));
    return pu::count_raw_errors(ctx, llr, llr_stride, n_bits, n_valid, coded, coded_stride, coded_index, bin, B, strong, counters,
                                reinterpret_cast<cudaStream_t>(stream));
}

pu_status pu_count_errors(pu_ctx* ctx, const uint8_t* info_bytes, size_t info_stride, const uint8_t* ok,
                          const int32_t* iters, const uint8_t* payload_pool, size_t payload_stride,
                          const uint32_t* tx_index, const uint32_t* bin, size_t payload_bytes, size_t B,
                          uint64_t* counters, void* stream) {
    PU_REQUIRE(ctx && info_bytes && ok && payload_pool && counters, "pu_count_errors: NULL argument");
    PU_REQUIRE(payload_bytes <= info_stride && payload_bytes <= payload_stride, "pu_count_errors: payload longer than its buffers");
    if (B == 0) return PU_OK;
    PU_CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    (void)cudaGetLastError();
    pu::count_errors_kernel<<<static_cast<unsigned>((B + 1023) / 1024), 1024, 0, st>>>(
        info_bytes, info_stride, ok, iters, payload_pool, payload_stride, tx_index, bin, static_cast<int>(payload_bytes), B,
        reinterpret_cast<unsigned long long*>(counters));
    ctx->launches.fetch_add(1);
    PU_CUDA_TRY(cudaGetLastError());
    return PU_OK;
}

pu_status pu_receive_decode_batch(pu_ofdm* ofdm, pu_ldpc* ldpc, const float* samples, size_t B, size_t L,
                                  int training_symbols, const float* cfo_hz, const float* cfo_phase,
                                  uint8_t* info_bytes, size_t info_stride, uint8_t* ok, int32_t* iters,
                                  pu_memspace space, void* stream) {
    PU_REQUIRE(ofdm && ldpc, "pu_receive_decode_batch: NULL handle");
    if (B == 0) return PU_OK;
    PU_REQUIRE(samples && info_bytes, "pu_receive_decode_batch: NULL data pointer");
    pu_ctx* ctx = pu_ofdm_context(ofdm);
    PU_CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = pu::pick_stream(ctx, stream, space);
    const size_t kb = static_cast<size_t>((pu_ldpc_info_bits(ldpc) + 7) / 8);
    PU_REQUIRE(info_stride >= kb, "pu_receive_decode_batch: info_stride too small");
    pu_status s;
    if (space == PU_MEM_DEVICE) {
        if ((s = ctx->d_aux.reserve(B * PU_LDPC_N * sizeof(float))) != PU_OK) return s;
        float* d_llr = static_cast<float*>(ctx->d_aux.ptr);
        const int n_sym_dev = static_cast<int>(L / static_cast<size_t>(pu_ofdm_symbol_samples(ofdm)));
        if (static_cast<size_t>(std::max(0, n_sym_dev - training_symbols)) * static_cast<size_t>(pu_ofdm_bits_per_symbol(ofdm)) < PU_LDPC_N)
            PU_CUDA_TRY(cudaMemsetAsync(d_llr, 0, B * PU_LDPC_N * sizeof(float), st));   // frames shorter than a codeword: erasures
        if ((s = pu_ofdm_presynced_batch(ofdm, samples, B, L, training_symbols, cfo_hz, cfo_phase, d_llr, PU_LDPC_N, nullptr,
                                         nullptr, PU_MEM_DEVICE, st)) != PU_OK) return s;
        return pu_ldpc_decode_batch(ldpc, d_llr, PU_LDPC_N, B, info_bytes, info_stride, ok, iters, PU_MEM_DEVICE, st);
    }
    // Host buffers: a two-lane pipeline.  Each slab of frames goes H2D -> demod -> LDPC -> D2H on its lane's own
    // stream, so the copy of slab i+1 overlaps the kernels and the read-back of slab i.  Samples that already live
    // in pinned (page-locked) memory are DMA'd straight from the caller's buffer; pageable samples are staged through
    // the lane's pinned buffer (that memcpy overlaps the other lane's GPU work).  Only info bytes / flags come back.
    cudaPointerAttributes attr{};
    const bool src_pinned = cudaPointerGetAttributes(&attr, samples) == cudaSuccess && attr.type == cudaMemoryTypeHost;
    (void)cudaGetLastError();
    const size_t slab = std::min<size_t>(B, 4096);
    const size_t iters_off = ((slab * kb + 15) / 16) * 16;
    const size_t out_bytes = iters_off + slab * sizeof(int32_t) + slab;
    if (stream) {   // order the lanes after work already queued on the caller's stream
        PU_CUDA_TRY(cudaEventRecord(ctx->pipe_ev, st));
        for (auto& sl : ctx->pipe) PU_CUDA_TRY(cudaStreamWaitEvent(sl.stream, ctx->pipe_ev, 0));
    }
    for (auto& sl : ctx->pipe) {
        // a previous call that failed half-way may have left copies or kernels of this lane in flight: its staging buffers are
        // about to be reused, so wait for them (a no-op when the lane is idle)
        PU_CUDA_TRY(cudaStreamSynchronize(sl.stream));
        sl.nb = 0;
        if ((s = sl.d_in.reserve(slab * (L + 2) * sizeof(float))) != PU_OK) return s;
        if (!src_pinned && (s = sl.h_in.reserve(slab * L * sizeof(float))) != PU_OK) return s;
        if ((s = sl.d_llr.reserve(slab * PU_LDPC_N * sizeof(float))) != PU_OK) return s;
        if ((s = sl.d_out.reserve(out_bytes + 64)) != PU_OK) return s;
        if ((s = sl.h_out.reserve(out_bytes + 64)) != PU_OK) return s;
    }
    const int n_sym = static_cast<int>(L / static_cast<size_t>(pu_ofdm_symbol_samples(ofdm)));
    const bool short_frames = static_cast<size_t>(std::max(0, n_sym - training_symbols)) *
                              static_cast<size_t>(pu_ofdm_bits_per_symbol(ofdm)) < PU_LDPC_N;
    auto drain = [&](pu::PipeSlot& sl) -> pu_status {
        if (sl.nb == 0) return PU_OK;
        PU_CUDA_TRY(cudaStreamSynchronize(sl.stream));
        const uint8_t* hout = static_cast<const uint8_t*>(sl.h_out.ptr);
        const int32_t* h_iters = reinterpret_cast<const int32_t*>(hout + iters_off);
        const uint8_t* h_ok = reinterpret_cast<const uint8_t*>(h_iters + slab);
        if (info_stride == kb) std::memcpy(info_bytes + sl.off * kb, hout, sl.nb * kb);
        else for (size_t b = 0; b < sl.nb; ++b) std::memcpy(info_bytes + (sl.off + b) * info_stride, hout + b * kb, kb);
        if (ok) std::memcpy(ok + sl.off, h_ok, sl.nb);
        if (iters) std::memcpy(iters + sl.off, h_iters, sl.nb * sizeof(int32_t));
        sl.nb = 0;
        return PU_OK;
    };
    size_t lane = 0;
    auto run = [&]() -> pu_status {
    for (size_t off = 0; off < B; off += slab, lane ^= 1) {
        pu::PipeSlot& sl = ctx->pipe[lane];
        if ((s = drain(sl)) != PU_OK) return s;
        const size_t nb = std::min(slab, B - off);
        cudaStream_t ls = sl.stream;
        float* din = static_cast<float*>(sl.d_in.ptr);
        const float* src = samples + off * L;
        // Zero-CFO 512-FFT differential frames go to the ofdm_diff512 kernel, which reads only the FFT windows of the symbols behind
        // the first training symbol: one strided (3-D) DMA moves exactly those (M1: 12 x 512 of 7 332 samples = 84 % of the frame);
        // the cyclic prefixes, guards and the first LTS symbol never cross PCIe.  Anything else is copied whole.
        int w_first = 0, w_nsym = 0, w_sym = 0, w_cp = 0, w_nfft = 0;
        const bool windowed = !cfo_hz && !cfo_phase &&
                              pu_ofdm_diff512_window(ofdm, din, nb, L, training_symbols, &w_first, &w_nsym, &w_sym, &w_cp, &w_nfft);
        if (!src_pinned) {   // pageable source: stage through the lane's pinned buffer (only the windows, when windowed)
            float* stage = static_cast<float*>(sl.h_in.ptr);
            if (windowed) {
                for (size_t b = 0; b < nb; ++b)
                    for (int sy = w_first; sy < w_nsym; ++sy) {
                        const size_t o = b * L + static_cast<size_t>(sy) * w_sym + w_cp;
                        std::memcpy(stage + o, src + o, static_cast<size_t>(w_nfft) * sizeof(float));
                    }
            } else {
                std::memcpy(stage, src, nb * L * sizeof(float));
            }
            src = stage;
        }
        if (windowed) {
            cudaMemcpy3DParms c3{};
            c3.srcPtr = make_cudaPitchedPtr(const_cast<float*>(src), static_cast<size_t>(w_sym) * sizeof(float), static_cast<size_t>(w_sym) * sizeof(float), static_cast<size_t>(w_nsym));
            c3.dstPtr = make_cudaPitchedPtr(din, static_cast<size_t>(w_sym) * sizeof(float), static_cast<size_t>(w_sym) * sizeof(float), static_cast<size_t>(w_nsym));
            c3.srcPos = make_cudaPos(static_cast<size_t>(w_cp) * sizeof(float), static_cast<size_t>(w_first), 0);
            c3.dstPos = c3.srcPos;
            c3.extent = make_cudaExtent(static_cast<size_t>(w_nfft) * sizeof(float), static_cast<size_t>(w_nsym - w_first), nb);
            c3.kind = cudaMemcpyHostToDevice;
            PU_CUDA_TRY(cudaMemcpy3DAsync(&c3, ls));
            ctx->h2d_bytes.fetch_add(static_cast<uint64_t>(nb) * (w_nsym - w_first) * w_nfft * sizeof(float));
        } else {
            PU_CUDA_TRY(cudaMemcpyAsync(din, src, nb * L * sizeof(float), cudaMemcpyHostToDevice, ls));
            ctx->h2d_bytes.fetch_add(static_cast<uint64_t>(nb) * L * sizeof(float) + (cfo_hz ? nb * sizeof(float) : 0) + (cfo_phase ? nb * sizeof(float) : 0));
        }
        const float *d_cfo = nullptr, *d_ph = nullptr;
        if (cfo_hz) {
            PU_CUDA_TRY(cudaMemcpyAsync(din + slab * L, cfo_hz + off, nb * sizeof(float), cudaMemcpyHostToDevice, ls));
            d_cfo = din + slab * L;
        }
        if (cfo_phase) {
            PU_CUDA_TRY(cudaMemcpyAsync(din + slab * L + slab, cfo_phase + off, nb * sizeof(float), cudaMemcpyHostToDevice, ls));
            d_ph = din + slab * L + slab;
        }
        float* d_llr = static_cast<float*>(sl.d_llr.ptr);
        if (short_frames) PU_CUDA_TRY(cudaMemsetAsync(d_llr, 0, nb * PU_LDPC_N * sizeof(float), ls));   // missing LLRs = erasures
        if ((s = pu_ofdm_presynced_batch(ofdm, din, nb, L, training_symbols, d_cfo, d_ph, d_llr, PU_LDPC_N, nullptr, nullptr,
                                         PU_MEM_DEVICE, ls)) != PU_OK) return s;
        uint8_t* d_info = static_cast<uint8_t*>(sl.d_out.ptr);
        int32_t* d_iters = reinterpret_cast<int32_t*>(d_info + iters_off);
        uint8_t* d_ok = reinterpret_cast<uint8_t*>(d_iters + slab);
        if ((s = pu_ldpc_decode_batch(ldpc, d_llr, PU_LDPC_N, nb, d_info, kb, d_ok, d_iters, PU_MEM_DEVICE, ls)) != PU_OK) return s;
        PU_CUDA_TRY(cudaMemcpyAsync(sl.h_out.ptr, d_info, out_bytes, cudaMemcpyDeviceToHost, ls));
        ctx->d2h_bytes.fetch_add(out_bytes);
        sl.off = off;
        sl.nb = nb;
    }
    if ((s = drain(ctx->pipe[lane])) != PU_OK) return s;
    if ((s = drain(ctx->pipe[lane ^ 1])) != PU_OK) return s;
    return PU_OK;
    };
    const pu_status rs = run();
    if (rs != PU_OK) {   // leave no lane in flight behind an error: the caller's buffers and the staging buffers must be quiescent
        for (auto& sl : ctx->pipe) { (void)cudaStreamSynchronize(sl.stream); sl.nb = 0; }
        (void)cudaGetLastError();
    }
    return rs;
}

}  // extern "C"
