// projectultra_b200/csrc/frame_v2.cu — protocol-v2 multi-codeword frames behind the batched decoder (SURVEY §8f next-4).
//
// Reference behaviour: RxPipeline::decodeFrame (src/gui/modem/rx_pipeline.cpp:348-445) over v2::decodeSingleCodeword
// (src/protocol/frame_v2.cpp:1134-1156), v2::parseHeader (:1175-1230, CRC-16/CCITT of :111-124), CodewordStatus::reassemble /
// reassembleCodewords (:952-982,1023-1044), and v2::encodeFrameWithLDPC (:1079-1127) on the transmit side.
// All codewords of all frames go through ONE launch of the LDPC kernel (the reference decodes CW1+ only once CW0 parses; decoding them
// anyway changes no result, the counters below follow the reference's control flow); a second kernel — one warp per frame — parses
// the header, applies the "enough codewords / all decoded" rules and reassembles the frame bytes.  Byte work, HBM-trivial.
#include <algorithm>
#include <cstring>
#include <vector>

#include "frame_v2.cuh"
#include "pu_internal.h"

namespace pu {

// info[b] = {success, frame_type, codewords_ok, codewords_failed, expected codewords}; frame_len[b] = bytes written to frame_out[b].
// Frame b owns ncw_stride codewords; it has ncw_b = ncw_per ? ncw_per[b] : ncw_stride of them (the soft bits an acquiring receiver
// delivered): codewords beyond ncw_b are never looked at.
__global__ void __launch_bounds__(128) frame_assemble_kernel(const uint8_t* __restrict__ cw_bytes, size_t cw_stride, const uint8_t* __restrict__ cw_ok,
                                                             int B, int ncw_stride, const int32_t* __restrict__ ncw_per, int bpc, int kbytes,
                                                             uint8_t* __restrict__ frame_out, size_t frame_cap, int32_t* __restrict__ frame_len,
                                                             int32_t* __restrict__ info) {
    const int lane = threadIdx.x & 31;
    const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (b >= B) return;
    const uint8_t* cw = cw_bytes + static_cast<size_t>(b) * ncw_stride * cw_stride;
    const uint8_t* ok = cw_ok + static_cast<size_t>(b) * ncw_stride;
    const int ncw = ncw_per ? min(ncw_per[b], ncw_stride) : ncw_stride;
    int success = 0, type = 0, n_ok = 0, n_fail = 0, expected = 0, out_len = 0;
    do {
        if (ncw < 1) break;                                              // soft_bits.size() < LDPC_BLOCK (:352-354)
        if (!ok[0] || kbytes < bpc) { n_fail = 1; break; }               // CW0 failed (:370-375)
        n_ok = 1;
        // parseHeader on lane 0, broadcast
        int valid = 0, is_control = 0, payload_len = 0;
        if (lane == 0) {
            const uint8_t* d = cw;
            if (((d[0] << 8) | d[1]) == 0x554C) {
                type = d[2];
                is_control = type == 0x10 || type == 0x11 || type == 0x16 || type == 0x17 || type == 0x20 || type == 0x21 || type == 0x40;
                if (is_control) {
                    valid = ((d[18] << 8) | d[19]) == frame_crc16(d, 18);
                    expected = 1;
                } else {
                    expected = d[12];
                    payload_len = (d[13] << 8) | d[14];
                    valid = ((d[15] << 8) | d[16]) == frame_crc16(d, 15);
                }
            }
        }
        valid = __shfl_sync(0xffffffffu, valid, 0);
        if (!valid) { type = 0; expected = 0; break; }                   // invalid header (:380-384)
        type = __shfl_sync(0xffffffffu, type, 0);
        is_control = __shfl_sync(0xffffffffu, is_control, 0);
        expected = __shfl_sync(0xffffffffu, expected, 0);
        payload_len = __shfl_sync(0xffffffffu, payload_len, 0);
        if (ncw < expected) break;                                       // waiting for more codewords (:394-401)
        for (int i0 = 1; i0 < expected; i0 += 32) {                      // CW1+ (:410-426)
            const int i = i0 + lane;
            const unsigned good = __ballot_sync(0xffffffffu, i < expected && ok[i]);
            const unsigned bad = __ballot_sync(0xffffffffu, i < expected && !ok[i]);
            n_ok += __popc(good);
            n_fail += __popc(bad);
        }
        if (n_fail) break;                                               // allSuccess (:429)
        success = 1;
        if (expected == 0) break;                                        // (undefined in the reference: it writes decoded[0] of an empty vector)
        // CodewordStatus::reassemble -> reassembleCodewords (frame_v2.cpp:952-982,1023-1044)
        const int expected_size = is_control ? 20 : 17 + payload_len + 2;
        uint8_t* out = frame_out + static_cast<size_t>(b) * frame_cap;
        int pos = 0;
        for (int i = 0; i < expected && pos < expected_size; ++i) {
            const uint8_t* src = cw + static_cast<size_t>(i) * cw_stride;
            int avail = bpc;
            if (i > 0 && src[0] == 0xD5) { src += 2; avail = bpc - 2; }  // marker + index skipped; otherwise the legacy fallback copies all
            const int take = min(expected_size - pos, avail);
            for (int j = lane; j < take; j += 32)
                if (static_cast<size_t>(pos + j) < frame_cap) out[pos + j] = src[j];
            pos += take;
        }
        out_len = pos;
    } while (false);
    if (lane == 0) {
        frame_len[b] = out_len;
        int32_t* o = info + static_cast<size_t>(b) * 5;
        o[0] = success; o[1] = type; o[2] = n_ok; o[3] = n_fail; o[4] = expected;
    }
}

pu_status frame_decode_enqueue(pu_ctx* ctx, pu_ldpc* dec, const float* llr, size_t B, int num_codewords, const int32_t* ncw_per,
                               uint8_t* cw_bytes, uint8_t* cw_ok, int32_t* cw_iters, uint8_t* frame_out, size_t frame_cap, int32_t* frame_len,
                               int32_t* info, cudaStream_t st) {
    const int kbytes = (pu_ldpc_info_bits(dec) + 7) / 8, bpc = frame_bytes_per_codeword(pu_ldpc_rate(dec));
    const pu_status s = pu_ldpc_decode_batch(dec, llr, PU_LDPC_N, B * static_cast<size_t>(num_codewords), cw_bytes, static_cast<size_t>(kbytes),
                                             cw_ok, cw_iters, PU_MEM_DEVICE, st);
    if (s != PU_OK) return s;
    const int warps = 4;
    (void)cudaGetLastError();
    frame_assemble_kernel<<<static_cast<unsigned>((B + warps - 1) / warps), warps * 32, 0, st>>>(
        cw_bytes, static_cast<size_t>(kbytes), cw_ok, static_cast<int>(B), num_codewords, ncw_per, bpc, kbytes, frame_out, frame_cap, frame_len, info);
    ctx->launches.fetch_add(1);
    PU_CUDA_TRY(cudaGetLastError());
    return PU_OK;
}

}  // namespace pu

extern "C" {

pu_status pu_frame_decode_batch(pu_ctx* ctx, pu_ldpc* dec, const float* llr, size_t B, size_t num_codewords, uint8_t* frame_out,
                                size_t frame_cap, int32_t* frame_len, int32_t* info, pu_memspace space, void* stream) {
    PU_REQUIRE(ctx && dec, "pu_frame_decode_batch: NULL handle");
    if (B == 0) return PU_OK;
    PU_REQUIRE(llr && frame_out && frame_len && info, "pu_frame_decode_batch: NULL data pointer");
    PU_REQUIRE(num_codewords >= 1 && num_codewords <= 255 && frame_cap > 0 && B * num_codewords < (1u << 30), "pu_frame_decode_batch: bad size");
    PU_CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = pu::pick_stream(ctx, stream, space);
    if (space == PU_MEM_HOST) {
        pu::HostStage hs(ctx, st, B);
        const float* d_llr;
        uint8_t* d_frame;
        int32_t *d_len, *d_info;
        hs.in(&d_llr, llr, num_codewords * PU_LDPC_N);
        hs.out(&d_frame, frame_out, frame_cap);
        hs.out(&d_len, frame_len, 1);
        hs.out(&d_info, info, 5);
        return hs.run([&](size_t nb) {
            return pu_frame_decode_batch(ctx, dec, d_llr, nb, num_codewords, d_frame, frame_cap, d_len, d_info, PU_MEM_DEVICE, st);
        });
    }
    const int kbytes = (pu_ldpc_info_bits(dec) + 7) / 8;
    const size_t ncw = B * num_codewords;
    // grow-only scratch on the context (the calling convention is one thread per context, as for the reference's objects)
    pu_status s;
    if ((s = ctx->f_bytes.reserve(ncw * static_cast<size_t>(kbytes))) != PU_OK) return s;
    if ((s = ctx->f_ok.reserve(ncw)) != PU_OK) return s;
    if ((s = ctx->f_iters.reserve(ncw * sizeof(int32_t))) != PU_OK) return s;
    s = pu::frame_decode_enqueue(ctx, dec, llr, B, static_cast<int>(num_codewords), nullptr, static_cast<uint8_t*>(ctx->f_bytes.ptr),
                                 static_cast<uint8_t*>(ctx->f_ok.ptr), static_cast<int32_t*>(ctx->f_iters.ptr), frame_out, frame_cap, frame_len, info, st);
    if (s != PU_OK) return s;
    PU_CUDA_TRY(cudaStreamSynchronize(st));           // results are complete on return (the scratch is reused by the next call)
    return PU_OK;
}

// v2::encodeFrameWithLDPC (frame_v2.cpp:1079-1127), host side: CW0 = the first bytes_per_cw frame bytes, CW1+ = {0xD5, index, payload},
// zero-padded, each LDPC-encoded to 81 bytes.  out == NULL queries the codeword count.
pu_status pu_frame_encode(int code_rate, const uint8_t* frame, size_t n_bytes, uint8_t* out, size_t out_cap, size_t* n_codewords) {
    PU_REQUIRE(n_codewords && (frame || n_bytes == 0), "pu_frame_encode: NULL argument");
    const size_t bpc = static_cast<size_t>(pu::frame_bytes_per_codeword(code_rate)), pay = bpc - 2;
    const size_t ncw = pu::frame_codewords(code_rate, n_bytes);
    *n_codewords = ncw;
    if (!out) return PU_OK;
    PU_REQUIRE(out_cap >= ncw * 81, "pu_frame_encode: output buffer too small");
    PU_REQUIRE(ncw <= 255, "pu_frame_encode: frame needs more than 255 codewords");
    std::vector<uint8_t> chunk(bpc);
    size_t offset = 0;
    for (size_t i = 0; i < ncw; ++i) {
        std::fill(chunk.begin(), chunk.end(), 0);
        if (i == 0) {
            std::memcpy(chunk.data(), frame, std::min(bpc, n_bytes));
            offset = bpc;
        } else {
            chunk[0] = 0xD5;
            chunk[1] = static_cast<uint8_t>(i);
            std::memcpy(chunk.data() + 2, frame + offset, std::min(pay, n_bytes - offset));
            offset += pay;
        }
        size_t len = 0;
        const pu_status s = pu_ldpc_encode(code_rate, chunk.data(), bpc, out + i * 81, 81, &len);
        if (s != PU_OK) return s;
    }
    return PU_OK;
}

}  // extern "C"
