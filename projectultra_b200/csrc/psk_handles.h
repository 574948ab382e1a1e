// projectultra_b200/csrc/psk_handles.h — handle types of the single-carrier / multi-carrier DPSK entry points, shared by
// psk_demod.cu (receive side) and psk_tx_gpu.cu (batched transmitters).
#pragma once
#include "pu_internal.h"

struct pu_dpsk {
    pu_ctx* ctx = nullptr;
    int device = 0;
    pu_dpsk_config cfg{};
    pu::DevMem d_cos, d_sin;
    pu::DevMem d_mf;        // matched-filter template of refineTimingWithMatchedFilter (cfo 0), 6 symbols
    float mf_energy = 0.0f;
    pu::Buffer corr;
    // batched transmitter (psk_tx_gpu.cu), built on first use: Barker preamble, carrier phase of every data sample, pulse shape
    pu::DevMem d_tx_pre, d_tx_phase, d_tx_pulse;
    size_t tx_pre_len = 0, tx_phase_syms = 0;
    float tx_symbol_phase0 = 0.0f;
};

struct pu_mcdpsk {
    pu_ctx* ctx = nullptr;
    int device = 0;
    pu_mcdpsk_config cfg{};
    pu::DevMem d_mixer, d_expected;
    pu::Buffer corr;
    pu::Buffer corrected;      // CFO-corrected copy of the batch (mcdpsk_got_chirp): kept between calls, grows on demand
    pu::DevMem d_chirp;     // dual-chirp templates (built on first use)
    pu::ChirpDev chirp{};
    bool chirp_ready = false;
    // batched transmitter (psk_tx_gpu.cu), built on first use: training + reference symbols, polar(1, i * inc_c) per (carrier, sample)
    pu::DevMem d_tx_pre, d_tx_polar;
    size_t tx_pre_len = 0;
    int tx_il_inv = 0;         // pu_mcdpsk_set_tx_interleave: step^-1 mod 648 of ChannelInterleaver, 0 = no interleaving
};

