// projectultra_b200/csrc/frame_v2.cuh — protocol-v2 frame layout shared by the host and the device: the CRC, the codeword chunking of
// v2::encodeFrameWithLDPC and the DATA-frame serialiser.  One definition serves the decoder (frame_v2.cu), the batched transmitter
// (ofdm_tx_gpu.cu), the sweep's host TX pool and its fresh-frame kernel (sweep.cu), so the frames they build cannot drift apart.
#pragma once
#include <cstdint>

#include "pu/pu_capi.h"

namespace pu {

__host__ __device__ inline uint16_t frame_crc16(const uint8_t* d, int len) {   // ControlFrame::calculateCRC, frame_v2.cpp:111-124
    uint16_t crc = 0xFFFF;
    for (int i = 0; i < len; ++i) {
        crc ^= static_cast<uint16_t>(static_cast<uint16_t>(d[i]) << 8);
        for (int j = 0; j < 8; ++j) crc = (crc & 0x8000) ? static_cast<uint16_t>((crc << 1) ^ 0x1021) : static_cast<uint16_t>(crc << 1);
    }
    return crc;
}

__host__ __device__ inline int frame_bytes_per_codeword(int rate) {   // getBytesPerCodeword, frame_v2.hpp:551-566
    switch (rate) {
        case PU_RATE_1_4: return 162 / 8;
        case PU_RATE_1_3: return 216 / 8;
        case PU_RATE_1_2: return 324 / 8;
        case PU_RATE_2_3: return 432 / 8;
        case PU_RATE_3_4: return 486 / 8;
        case PU_RATE_5_6: return 540 / 8;
        default: return 162 / 8;
    }
}

// codewords of an n_bytes frame: CW0 carries bpc bytes, CW1+ bpc - 2 behind their {0xD5, index} prefix (encodeFrameWithLDPC,
// frame_v2.cpp:1079-1127; the same count as DataFrame::calculateCodewords, :439-460, writes into TOTAL_CW)
__host__ __device__ inline uint64_t frame_codewords(int rate, uint64_t n_bytes) {
    const uint64_t bpc = static_cast<uint64_t>(frame_bytes_per_codeword(rate)), pay = bpc - 2;
    return n_bytes <= bpc ? 1 : 1 + (n_bytes - bpc + pay - 1) / pay;
}

constexpr int kV2DataHeader = 17;      // DATA header: magic, type, flags, seq, src, dst, TOTAL_CW, payload length, header CRC
constexpr int kV2FrameOverhead = 19;   // ... plus the frame CRC behind the payload

// DataFrame::serialize (frame_v2.cpp:502-555) IN PLACE: the payload already sits at frame[17 .. 17 + payload_len); writes the header in
// front of it and the frame CRC behind it (frame[0 .. payload_len + 19)).  The sweep's frames carry src 0x123456, dst 0xABCDEF,
// type 0x30 and flags 0x01 (linksim.v2_data_frame's defaults).
__host__ __device__ inline void v2_data_frame_in_place(uint8_t* frame, int payload_len, int rate, uint16_t seq) {
    const uint32_t src = 0x123456u, dst = 0xABCDEFu;
    const int tcw = static_cast<int>(frame_codewords(rate, static_cast<uint64_t>(payload_len) + kV2FrameOverhead));
    const uint8_t h[15] = {0x55, 0x4C, 0x30, 0x01, static_cast<uint8_t>(seq >> 8), static_cast<uint8_t>(seq & 0xFF),
                           static_cast<uint8_t>(src >> 16), static_cast<uint8_t>((src >> 8) & 0xFF), static_cast<uint8_t>(src & 0xFF),
                           static_cast<uint8_t>(dst >> 16), static_cast<uint8_t>((dst >> 8) & 0xFF), static_cast<uint8_t>(dst & 0xFF),
                           static_cast<uint8_t>(tcw), static_cast<uint8_t>(payload_len >> 8), static_cast<uint8_t>(payload_len & 0xFF)};
    for (int i = 0; i < 15; ++i) frame[i] = h[i];
    const uint16_t hc = frame_crc16(frame, 15);
    frame[15] = static_cast<uint8_t>(hc >> 8);
    frame[16] = static_cast<uint8_t>(hc & 0xFF);
    const int body = kV2DataHeader + payload_len;
    const uint16_t fc = frame_crc16(frame, body);
    frame[body] = static_cast<uint8_t>(fc >> 8);
    frame[body + 1] = static_cast<uint8_t>(fc & 0xFF);
}

}  // namespace pu
