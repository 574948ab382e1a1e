// projectultra_b200/csrc/ldpc_encode.cuh — v2::encodeFrameWithLDPC chunking + LDPCEncoder::encode of a whole frame by one CTA, into a
// buffer the CTA owns (shared memory).  One definition serves the batched OFDM transmitter (ofdm_tx_gpu.cu) and the batched encoder
// behind pu_ldpc_encode_batch / pu_frame_encode_batch (ldpc_encode.cu), so the coded bits they produce cannot drift apart.
//
//   v2::encodeFrameWithLDPC (chunking)                    src/protocol/frame_v2.cpp:1079-1127
//   LDPCEncoder::encode                                   src/fec/ldpc_encoder.cpp:193-257  (parity_i = XOR of H_data row i)
#pragma once
#include <cstdint>

#include "pu/pu_capi.h"

namespace pu {

// LDPC tables in slot order (ldpc_code.h: LdpcHostTables), as pu_ldpc_encoder_view hands them out
struct LdpcEncDev {
    int k, m;
    const uint8_t* cn_ninfo;
    const uint16_t* cn_check;
    const uint16_t* cn_var;
};

// Bytes the encoder needs per CTA: the n_cw * 81 coded bytes packed MSB first, then the inverse of the parity placement.
inline size_t ldpc_encode_smem(int n_cw, int m) { return static_cast<size_t>(n_cw) * (PU_LDPC_N / 8) + static_cast<size_t>(m) * sizeof(uint16_t) + 16; }
__device__ inline uint16_t* ldpc_encode_parity_of(uint8_t* smem, int n_cw) {
    return reinterpret_cast<uint16_t*>(smem + ((static_cast<size_t>(n_cw) * (PU_LDPC_N / 8) + 1) & ~size_t(1)));
}

// The frame fr[0 .. frame_bytes) -> coded[n_cw][81].  CW0 = frame bytes [0, bpc), CWi = {0xD5, i, bytes [bpc + (i-1)(bpc-2), ...)}, zero
// padded to the codeword's k information bits (bpc * 8 <= k; the bits from bpc * 8 to k are zero), then parity bit r = XOR of H_data row
// parity_of[r].  Every thread of the CTA calls it; it ends on a barrier, after which coded[] is complete.
__device__ inline void ldpc_encode_frame_cta(const LdpcEncDev& e, const uint8_t* __restrict__ fr, int frame_bytes, int n_cw, int bpc,
                                             uint8_t* coded, uint16_t* parity_of) {
    constexpr int kCwBytes = PU_LDPC_N / 8;               // 648 = 81 bytes exactly: codewords stay byte aligned back to back
    const int tid = threadIdx.x, T = blockDim.x;
    for (int j = tid; j < n_cw * bpc; j += T) {
        const int i = j / bpc, q = j - i * bpc;
        int src = q;
        uint8_t v;
        if (i == 0) v = q < frame_bytes ? fr[q] : 0;
        else if (q < 2) v = q == 0 ? 0xD5 : static_cast<uint8_t>(i);
        else { src = bpc + (i - 1) * (bpc - 2) + q - 2; v = src < frame_bytes ? fr[src] : 0; }
        coded[i * kCwBytes + q] = v;
    }
    for (int p = tid; p < e.m; p += T) parity_of[e.cn_check[p]] = static_cast<uint16_t>(p);
    __syncthreads();
    // one thread per output byte from byte bpc on (whole bytes, so no two threads write one byte)
    const int info_bits = bpc * 8;
    for (int j = tid; j < n_cw * (kCwBytes - bpc); j += T) {
        const int i = j / (kCwBytes - bpc), q = bpc + (j - i * (kCwBytes - bpc));
        const uint8_t* cw = coded + i * kCwBytes;
        unsigned byte = 0;
        for (int b = 0; b < 8; ++b) {
            const int bit = q * 8 + b;
            unsigned acc = 0;
            if (bit >= e.k) {
                const int p = parity_of[bit - e.k];
                const int ninfo = e.cn_ninfo[p];
                for (int x = 0; x < ninfo; ++x) {
                    const int v = e.cn_var[x * e.m + p];
                    if (v < info_bits) acc ^= (cw[v >> 3] >> (7 - (v & 7))) & 1u;
                }
            }
            byte = (byte << 1) | acc;
        }
        coded[i * kCwBytes + q] = static_cast<uint8_t>(byte);
    }
    __syncthreads();
}

}  // namespace pu
