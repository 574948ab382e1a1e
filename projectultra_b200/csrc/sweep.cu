// projectultra_b200/csrc/sweep.cu — the Monte-Carlo sweep driver behind the C ABI (pu_linksim_run, pu_sweep_*, pu_counters_allreduce):
// BASELINE.json config 5, "full adaptive-mode FER/BER waterfall (all waveforms x rates x SNR points x seeds) sharded across 8 GPUs".
//
// Host logic only (C++20); every sample is produced and consumed by the kernels behind the other C-ABI entry points, which this file
// calls with device pointers on the context's stream.  The reference's shape is a shell matrix over one-process-per-cell tools
// (tests/regression_matrix.sh:139-243, tools/test_iwaveform.cpp:597-806, tools/test_mode_snr.cpp:40-105); see pu_capi.h for the
// contract.  Work units (mode, SNR point, seed block) -> ranks by longest-processing-time-first on a cost estimate; a rank runs its
// units mode by mode in batches that mix SNR points and seed blocks (counter bin = unit), two batches in flight so that descriptor
// preparation and the manifest append of batch k overlap the kernels of batch k+1.  Frame modes (pu_sweep_mode.frame_payload_bytes) carry
// a protocol-v2 DATA frame of several codewords per trial (v2::encodeFrameWithLDPC, frame_v2.cpp:1079-1127) and count whole frames as
// RxPipeline::decodeFrame (rx_pipeline.cpp:348-445) delivers them.
#include <dlfcn.h>
#include <sys/stat.h>
#include <dirent.h>
#include <unistd.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <memory>
#include <numeric>
#include <queue>
#include <string>
#include <vector>

#include "frame_v2.cuh"
#include "ofdm_plan.h"
#include "pu_internal.h"

namespace pu {
namespace {

constexpr uint32_t kNoOwner = 0xffffffffu;

struct SweepPlan {
    uint32_t pool, block, max_iter;
    uint64_t base_seed, trials, batch_bytes;
    std::vector<uint64_t> unit0;      // first unit id of mode m (size n_modes + 1)
    std::vector<uint32_t> point0;     // first counter row of mode m (size n_modes + 1)
    uint64_t blocks;                  // seed blocks per (mode, SNR point)
    std::vector<uint32_t> n_cw;       // codewords per trial of mode m (1 in codeword mode)
    std::vector<double> frame_scale;  // OFDM symbols of a frame of mode m over those of a one-codeword frame (1 in codeword mode)
};

// frame mode (pu_sweep_mode.frame_payload_bytes): the OFDM waveforms only, DataFrame::serialize's 16-bit length, at most the 255
// codewords TOTAL_CW can count.  n_cw and the frame's length in OFDM symbols relative to one codeword's (for the partitioner's cost).
bool frame_mode_shape(const pu_sweep_mode& md, uint32_t* n_cw, double* scale) {
    *n_cw = 1;
    *scale = 1.0;
    if (!md.frame_payload_bytes) return true;
    if (md.waveform > PU_WF_OFDM_CHIRP || md.frame_payload_bytes > 65535) return false;
    const uint64_t ncw = frame_codewords(static_cast<int>(md.code_rate), uint64_t(md.frame_payload_bytes) + kV2FrameOverhead);
    if (ncw > 255) return false;
    OfdmPlan plan;
    const char* why = "";
    if (!make_ofdm_plan(md.ofdm, &plan, &why)) return false;
    const uint64_t per_sym = static_cast<uint64_t>(plan.n_data) * plan.bps;
    *n_cw = static_cast<uint32_t>(ncw);
    *scale = (2.0 + static_cast<double>((ncw * PU_LDPC_N + per_sym - 1) / per_sym)) / (2.0 + static_cast<double>((PU_LDPC_N + per_sym - 1) / per_sym));
    return true;
}

bool make_plan(const pu_sweep_desc* d, SweepPlan* p) {
    if (!d || !d->modes || d->n_modes == 0 || d->trials_per_point == 0 || d->world == 0 || d->rank >= d->world) return false;
    p->pool = d->pool ? d->pool : 64;
    p->block = d->block_trials ? d->block_trials : 4096;
    p->max_iter = d->max_iter ? d->max_iter : 50;
    p->base_seed = d->base_seed ? d->base_seed : 0xB200;
    p->trials = d->trials_per_point;
    p->batch_bytes = d->batch_bytes ? d->batch_bytes : (uint64_t(3) << 29);
    p->blocks = (p->trials + p->block - 1) / p->block;
    p->unit0.assign(1, 0);
    p->point0.assign(1, 0);
    for (uint32_t m = 0; m < d->n_modes; ++m) {
        const pu_sweep_mode& md = d->modes[m];
        if (md.n_snr == 0 || md.n_snr > 255 || md.waveform > PU_WF_MCDPSK_CHIRP || md.channel > PU_CH_ITU_FLUTTER) return false;
        // ChannelInterleaver rides on the IWaveform path (OFDM, MC-DPSK); single-carrier DPSK has no interleaver in the reference
        if (md.interleave_bps && (md.waveform == PU_WF_DPSK || md.waveform == PU_WF_DPSK_ACQ)) return false;
        uint32_t ncw;
        double scale;
        if (!frame_mode_shape(md, &ncw, &scale)) return false;
        p->n_cw.push_back(ncw);
        p->frame_scale.push_back(scale);
        p->unit0.push_back(p->unit0.back() + static_cast<uint64_t>(md.n_snr) * p->blocks);
        p->point0.push_back(p->point0.back() + md.n_snr);
    }
    return d->n_modes <= 255;
}

// Built-in relative cost of one frame (GPU time, arbitrary unit), from the measured throughputs of DESIGN.md §4: the 512-FFT
// differential kernels run ~100 M frames/s, the general presynced kernel 10-30 M, Schmidl-Cox acquisition 0.3 M, Barker acquisition
// 0.25 M (139 392-sample frames), the two-tier dual-chirp search 0.34 M (OFDM_CHIRP) / 0.18 M (MC-DPSK, 84 200 samples), plus the
// channel kernel's share for these long frames; LDPC is
// added per SNR point by unit_cost().
double mode_cost(const pu_sweep_mode& m) {
    if (m.cost > 0) return m.cost;
    switch (m.waveform) {
        case PU_WF_OFDM: {
            const bool diff = m.ofdm.modulation == PU_MOD_DBPSK || m.ofdm.modulation == PU_MOD_DQPSK || m.ofdm.modulation == PU_MOD_D8PSK;
            return (diff && !m.ofdm.use_pilots && m.ofdm.fft_size == 512) ? 1.0 : (diff && !m.ofdm.use_pilots) ? 2.0 : 8.0;
        }
        case PU_WF_OFDM_SC: return 250.0;
        case PU_WF_OFDM_CHIRP: return 350.0;
        case PU_WF_DPSK: return 30.0;
        case PU_WF_DPSK_ACQ: return 480.0;
        case PU_WF_MCDPSK: return 10.0;
        default: return 620.0;      // PU_WF_MCDPSK_CHIRP
    }
}
// LDPC share: ~50 iterations at the bottom of the grid, ~2 at the top; in units of the demodulator cost of the cheapest mode
// (0.87 ms LDPC against 0.37 ms demod per 53 248 frames at 17 average iterations: ~0.14 per iteration).  A frame-mode trial costs
// its frame's length in demodulation and n_cw codewords in LDPC.
double unit_cost(const SweepPlan& p, const pu_sweep_mode& m, uint32_t mode, uint32_t snr_index, uint32_t n_trials) {
    const double f = m.n_snr > 1 ? 1.0 - static_cast<double>(snr_index) / (m.n_snr - 1) : 0.5;
    const double iters = 2.0 + 48.0 * f * f;
    const double demod = m.cost > 0 ? m.cost : mode_cost(m) * p.frame_scale[mode];      // a table's own cost is per trial already
    return n_trials * (demod + 0.14 * iters * p.n_cw[mode]);
}

void unit_decode(const pu_sweep_desc* d, const SweepPlan& p, uint64_t u, uint32_t* mode, uint32_t* snr, uint64_t* t0, uint32_t* nt) {
    uint32_t m = static_cast<uint32_t>(std::upper_bound(p.unit0.begin(), p.unit0.end(), u) - p.unit0.begin()) - 1;
    const uint64_t r = u - p.unit0[m];
    const uint32_t s = static_cast<uint32_t>(r / p.blocks);
    const uint64_t b = r % p.blocks;
    *mode = m; *snr = s; *t0 = b * p.block;
    *nt = static_cast<uint32_t>(std::min<uint64_t>(p.block, p.trials - *t0));
    (void)d;
}

uint64_t splitmix64(uint64_t& x) {
    uint64_t z = (x += 0x9e3779b97f4a7c15ull);
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
    return z ^ (z >> 31);
}

// FNV-1a over everything that defines the frames of a unit, and the record format: a raw run (pu_linksim_run_raw) mixes in one more tag,
// so that it and a plain run of the same table never resume from each other's shards; a plain run keeps the key its manifests have
uint64_t desc_key(const pu_sweep_desc* d, const SweepPlan& p, bool raw) {
    uint64_t h = 0xcbf29ce484222325ull;
    auto mix = [&h](const void* ptr, size_t n) {
        const unsigned char* b = static_cast<const unsigned char*>(ptr);
        for (size_t i = 0; i < n; ++i) { h ^= b[i]; h *= 0x100000001b3ull; }
    };
    mix(&d->n_modes, sizeof d->n_modes);
    for (uint32_t m = 0; m < d->n_modes; ++m) {
        pu_sweep_mode md = d->modes[m];
        md.cost = 0;             // the partitioner's weights do not change what a unit computes
        // fields appended to the mode enter the key only when set: a table without them keeps the key -- and the manifests -- it had
        mix(&md, offsetof(pu_sweep_mode, interleave_bps));
        if (md.interleave_bps) mix(&md.interleave_bps, sizeof md.interleave_bps);
    }
    mix(&p.pool, sizeof p.pool); mix(&p.block, sizeof p.block); mix(&p.max_iter, sizeof p.max_iter);
    mix(&p.base_seed, sizeof p.base_seed); mix(&p.trials, sizeof p.trials);
    if (raw) mix("raw counters", 12);
    return h;
}

// fresh_payloads: byte i of frame b's payload = byte (i & 7) of splitmix64(seed[b] ^ kPayloadStream ^ (i >> 3) * golden ratio); rows are kb bytes,
// zero past payload_bytes.  The frame seed also drives the channel; the stream constant keeps the two independent.
__device__ inline uint64_t fresh_payload_word(uint64_t seed, size_t w) {
    uint64_t z = (seed ^ 0x5041594c4f414421ull) + 0x9e3779b97f4a7c15ull * (w + 1);
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
    return z ^ (z >> 31);
}
__global__ void fresh_payload_kernel(uint8_t* __restrict__ pay, size_t kb, uint32_t payload_bytes, const uint64_t* __restrict__ seed, size_t B) {
    const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
    const size_t words = (kb + 7) / 8;
    if (i >= B * words) return;
    const size_t b = i / words, w = i - b * words;
    const uint64_t z = fresh_payload_word(seed[b], w);
    for (size_t k = 0; k < 8 && 8 * w + k < kb; ++k) pay[b * kb + 8 * w + k] = 8 * w + k < payload_bytes ? static_cast<uint8_t>(z >> (8 * k)) : 0;
}

// frame modes: row b of frames[B][stride] = the DATA frame around the same payload byte stream (payload_bytes bytes at offset 17), seq =
// the low 16 bits of the frame seed (= trial & 0xFFFF); one warp per frame, lane 0 serialises header and CRCs
__global__ void fresh_frame_kernel(uint8_t* __restrict__ frames, size_t stride, uint32_t payload_bytes, int rate, const uint64_t* __restrict__ seed, size_t B) {
    const int lane = threadIdx.x & 31;
    const size_t b = blockIdx.x * static_cast<size_t>(blockDim.x >> 5) + (threadIdx.x >> 5);
    if (b >= B) return;
    uint8_t* f = frames + b * stride;
    const uint64_t sd = seed[b];
    for (size_t w = lane; w < (payload_bytes + 7) / 8; w += 32) {
        const uint64_t z = fresh_payload_word(sd, w);
        for (size_t k = 0; k < 8 && 8 * w + k < payload_bytes; ++k) f[kV2DataHeader + 8 * w + k] = static_cast<uint8_t>(z >> (8 * k));
    }
    __syncwarp();
    if (lane == 0) v2_data_frame_in_place(f, static_cast<int>(payload_bytes), rate, static_cast<uint16_t>(sd & 0xFFFF));
}

// frame modes behind an acquiring receiver: the codewords of frame b that RxPipeline::decodeFrame gets = whole codewords of soft bits
// (0 without sync); codewords past them are never decoded into the result (an all-zero LLR block would "decode" to zeros)
__global__ void frame_codewords_kernel(int32_t* __restrict__ ncw, const int32_t* __restrict__ n_llr, int n_cw, size_t B) {
    const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
    if (i < B) ncw[i] = min(n_cw, max(0, n_llr[i]) / PU_LDPC_N);
}

// fresh payloads behind the chirp pair, one CTA per row: the pair into [lead, lead + chirp_len), then the tools' peak normalisation
// w * (peak / max|w|) over chirp and body together -- the order of the host pool (ModeEngine::build)
__global__ void chirp_peak_kernel(float* __restrict__ tx, size_t L, size_t lead, const float* __restrict__ chirp, size_t chirp_len, size_t body_len, float peak) {
    __shared__ float red[32];
    float* row = tx + blockIdx.x * L + lead;
    const size_t len = chirp_len + body_len;
    float mx = 0.0f;
    for (size_t i = threadIdx.x; i < len; i += blockDim.x) {
        const float v = i < chirp_len ? chirp[i] : row[i];
        if (i < chirp_len) row[i] = v;
        mx = fmaxf(mx, fabsf(v));
    }
    if (peak <= 0.0f) return;
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
    __syncthreads();
    mx = red[0];
    for (unsigned w = 1; w < blockDim.x / 32; ++w) mx = fmaxf(mx, red[w]);
    const float g = __fdiv_rn(peak, mx);
    for (size_t i = threadIdx.x; i < len; i += blockDim.x) row[i] = __fmul_rn(row[i], g);
}

__global__ void mask_short_kernel(uint8_t* __restrict__ ok, const int32_t* __restrict__ n_llr, size_t B) {
    // no sync / fewer than one codeword of soft bits is a lost frame (tools/test_mode_snr.cpp:72-77): override the decoder's verdict
    const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
    if (i < B && n_llr[i] < PU_LDPC_N) ok[i] = 0;
}

// ---- one mode of the table, instantiated on this rank ---------------------------------------------------------------------------
struct ModeEngine {
    pu_ctx* ctx = nullptr;
    const pu_sweep_mode* md = nullptr;
    pu_ofdm* ofdm = nullptr;
    pu_dpsk* dpsk = nullptr;
    pu_mcdpsk* mcd = nullptr;
    pu_ldpc* ldpc = nullptr;
    bool own_ldpc = true;                // false: the decoder of this code rate is shared by the run (pu_linksim_run keeps one per rate)
    pu_channel_config ch{};
    size_t L = 0, kb = 0;
    uint32_t pool = 0;
    int convention = 0;
    std::vector<float> noise_std;        // [n_snr][pool]; fresh payloads: [n_snr] SNR factors of pu_channel_noise_std_batch
    Buffer d_tx, d_payload;              // [pool][L] floats, [pool][kb] bytes
    Buffer d_coded;                      // raw counts: [pool][n_cw * 81] coded bytes of the pool, before interleaving
    bool fresh = false;                  // pu_sweep_mode.fresh_payloads: TX inside the batch
    size_t body_len = 0;                 // samples the transmitter writes per frame (L = lead + chirp + body + tail)
    size_t chirp_len = 0;                // fresh payloads of the chirp waveforms: the pair in d_chirp, written in front of every body
    Buffer d_chirp;
    pu_tools_cfo* tools_cfo = nullptr;   // fresh payloads with cfo_hz: the tools' injector over every row
    bool frames = false;                 // pu_sweep_mode.frame_payload_bytes > 0: a protocol-v2 DATA frame per trial
    uint32_t n_cw = 1;                   // codewords per trial
    size_t frame_bytes = 0;              // frame modes: bytes of the DATA frame (payload + 19)
    size_t pay_stride = 0;               // bytes per row of d_payload / the fresh payload rows: kb, or frame_bytes in frame modes
    bool deinterleave = false;           // pu_sweep_mode.interleave_bps on a receiver without the fused table: pu_llr_deinterleave_batch

    ~ModeEngine() {
        if (ofdm) pu_ofdm_destroy(ofdm);
        if (dpsk) pu_dpsk_destroy(dpsk);
        if (mcd) pu_mcdpsk_destroy(mcd);
        if (ldpc && own_ldpc) pu_ldpc_destroy(ldpc);
        if (tools_cfo) pu_tools_cfo_destroy(tools_cfo);
        d_tx.release(); d_payload.release(); d_chirp.release(); d_coded.release();
    }

    pu_status build(pu_ctx* c, const pu_sweep_mode* m, uint32_t mode_index, const SweepPlan& p, cudaStream_t st, pu_ldpc* shared_ldpc, bool raw) {
        ctx = c; md = m; pool = p.pool;
        pu_status s;
        const bool trace = std::getenv("PU_SWEEP_TRACE") != nullptr;
        auto now = [] { return std::chrono::steady_clock::now(); };
        auto secs = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) { return std::chrono::duration<double>(b - a).count(); };
        const auto t0 = now();
        if ((s = pu_channel_preset(static_cast<int>(m->channel), &ch)) != PU_OK) return s;
        // AWGN tools define SNR on mean frame power, WattersonChannel on input rms (same number, different rounding)
        convention = m->channel == PU_CH_AWGN ? 1 : 0;
        if (shared_ldpc) { ldpc = shared_ldpc; own_ldpc = false; }
        else if ((s = pu_ldpc_create(c, static_cast<int>(m->code_rate), static_cast<int>(p.max_iter), &ldpc)) != PU_OK) return s;
        const auto t_ldpc = now();
        kb = static_cast<size_t>((pu_ldpc_info_bits(ldpc) + 7) / 8);
        frames = m->frame_payload_bytes != 0;
        if (frames) {
            frame_bytes = m->frame_payload_bytes + kV2FrameOverhead;
            n_cw = static_cast<uint32_t>(frame_codewords(static_cast<int>(m->code_rate), frame_bytes));
        } else {
            PU_REQUIRE(m->payload_bytes >= 1 && m->payload_bytes <= kb, "pu_linksim_run: payload_bytes exceeds the code's information bytes");
        }
        pay_stride = frames ? frame_bytes : kb;
        const bool is_ofdm = m->waveform <= PU_WF_OFDM_CHIRP, is_dpsk = m->waveform == PU_WF_DPSK || m->waveform == PU_WF_DPSK_ACQ;
        if (is_ofdm) {
            if ((s = pu_ofdm_create(c, &m->ofdm, &ofdm)) != PU_OK) return s;
            if ((s = pu_ofdm_set_precision(ofdm, m->precision ? PU_PRECISION_FAST : PU_PRECISION_EXACT)) != PU_OK) return s;
        } else if (is_dpsk) {
            if ((s = pu_dpsk_create(c, &m->dpsk, &dpsk)) != PU_OK) return s;
        } else {
            if ((s = pu_mcdpsk_create(c, &m->mcdpsk, &mcd)) != PU_OK) return s;
        }
        if (m->interleave_bps) {
            // one deinterleaver per handle: the fused table of the presynced receiver only holds the first codeword of a row
            if (m->waveform != PU_WF_OFDM || frames) deinterleave = true;
            else if ((s = pu_ofdm_set_deinterleave(ofdm, m->interleave_bps, PU_LDPC_N)) != PU_OK) return s;
            if ((s = ofdm ? pu_ofdm_set_tx_interleave(ofdm, m->interleave_bps) : pu_mcdpsk_set_tx_interleave(mcd, m->interleave_bps)) != PU_OK) return s;
        }
        const auto t1 = now();
        const float fs = is_ofdm ? static_cast<float>(m->ofdm.sample_rate) : is_dpsk ? m->dpsk.sample_rate : m->mcdpsk.sample_rate;
        std::vector<float> chirp;             // the pair does not depend on the payload (tx_cfo_hz for OFDM, 0 for MC-DPSK)
        if (m->waveform == PU_WF_OFDM_CHIRP || m->waveform == PU_WF_MCDPSK_CHIRP) {
            size_t n = 0;
            pu_chirp_generate(fs, is_ofdm ? m->ofdm.tx_cfo_hz : 0.0f, nullptr, 0, &n);
            chirp.resize(n);
            if ((s = pu_chirp_generate(fs, is_ofdm ? m->ofdm.tx_cfo_hz : 0.0f, chirp.data(), n, &n)) != PU_OK) return s;
        }
        fresh = m->fresh_payloads != 0;
        if (fresh) {
            if ((s = tx_batch(nullptr, 0, nullptr, 0, st)) != PU_OK) return s;      // queries body_len
            chirp_len = chirp.size();
            L = m->lead_samples + chirp_len + body_len + m->tail_samples;
            if (chirp_len) {
                if ((s = d_chirp.reserve(chirp_len * sizeof(float))) != PU_OK) return s;
                PU_CUDA_TRY(cudaMemcpyAsync(d_chirp.ptr, chirp.data(), chirp_len * sizeof(float), cudaMemcpyHostToDevice, st));
                PU_CUDA_TRY(cudaStreamSynchronize(st));       // `chirp` is pageable and goes out of scope
            }
            if (m->cfo_hz != 0.0f && (s = pu_tools_cfo_create(c, L, m->cfo_hz, fs, &tools_cfo)) != PU_OK) return s;
            noise_std.resize(m->n_snr);
            for (uint32_t si = 0; si < m->n_snr; ++si) {
                const float snr = m->snr_first_db + si * m->snr_step_db;
                noise_std[si] = convention == 0 ? std::pow(10.0f, -snr / 20.0f) : std::pow(10.0f, snr / 10.0f);   // pu_channel_noise_std's factors
            }
            if (trace) fprintf(stderr, "[engine] mode %u: fresh payloads, %zu samples per frame\n", mode_index, L);
            return PU_OK;
        }
        // TX pool on the host (the reference's modulators run per trial on the CPU too): payload -> LDPC encode -> modulate [-> chirp in front]
        std::vector<std::vector<float>> waves(pool);
        // (frame modes: the payload inside DataFrame::serialize, seq i + 1 -> v2::encodeFrameWithLDPC -> all codewords modulated)
        std::vector<uint8_t> payloads(static_cast<size_t>(pool) * pay_stride, 0);
        std::vector<uint8_t> coded(static_cast<size_t>(n_cw) * (PU_LDPC_N / 8));
        std::vector<uint8_t> coded_pool(raw ? static_cast<size_t>(pool) * coded.size() : 0);
        for (uint32_t i = 0; i < pool; ++i) {
            uint8_t* pay = payloads.data() + static_cast<size_t>(i) * pay_stride;
            size_t nc = 0;
            if (frames) {
                pu_sweep_payload(p.base_seed, mode_index, i, pay + kV2DataHeader, m->frame_payload_bytes);
                v2_data_frame_in_place(pay, static_cast<int>(m->frame_payload_bytes), static_cast<int>(m->code_rate), static_cast<uint16_t>(i + 1));
                if ((s = pu_frame_encode(static_cast<int>(m->code_rate), pay, frame_bytes, coded.data(), coded.size(), &nc)) != PU_OK) return s;
                PU_REQUIRE(nc == n_cw, "pu_linksim_run: frame codeword count differs from the plan");
                nc *= PU_LDPC_N / 8;
            } else {
                pu_sweep_payload(p.base_seed, mode_index, i, pay, m->payload_bytes);
                if ((s = pu_ldpc_encode(static_cast<int>(m->code_rate), pay, m->payload_bytes, coded.data(), coded.size(), &nc)) != PU_OK) return s;
            }
            if (raw) std::copy(coded.begin(), coded.end(), coded_pool.begin() + static_cast<size_t>(i) * coded.size());
            if (m->interleave_bps) channel_interleave_codewords(m->interleave_bps, coded.data(), nc / (PU_LDPC_N / 8));
            size_t n = 0;
            std::vector<float> w;
            auto tx = [&](float* out, size_t cap, size_t* len) -> pu_status {
                if (is_ofdm) return pu_ofdm_tx(&m->ofdm, m->waveform == PU_WF_OFDM_SC ? 1 : 0, coded.data(), nc, out, cap, len);
                if (is_dpsk) return pu_dpsk_tx(&m->dpsk, 0, coded.data(), nc, out, cap, len);
                return pu_mcdpsk_tx(&m->mcdpsk, coded.data(), nc, out, cap, len);
            };
            // every waveform of a mode has the same length: the host modulators are asked for it once (a query runs the whole modulation)
            if (body_len == 0) { tx(nullptr, 0, &n); body_len = n; }
            w.resize(body_len);
            if ((s = tx(w.data(), body_len, &n)) != PU_OK) return s;
            PU_REQUIRE(n == body_len, "pu_linksim_run: TX waveforms of one mode differ in length");
            if (!chirp.empty()) w.insert(w.begin(), chirp.begin(), chirp.end());
            if (m->lead_samples) w.insert(w.begin(), m->lead_samples, 0.0f);       // the tools' silence around a frame (test_iwaveform.cpp:396-459)
            if (m->tail_samples) w.insert(w.end(), m->tail_samples, 0.0f);
            if (m->peak > 0) {
                float mx = 0.0f;
                for (float v : w) mx = std::max(mx, std::fabs(v));
                const float g = m->peak / mx;
                for (float& v : w) v *= g;
            }
            if (m->cfo_hz != 0.0f) tools_apply_cfo(w.data(), w.size(), m->cfo_hz, fs);   // the tools' --cfo: the clean audio, before the channel (test_iwaveform.cpp:501-506)
            waves[i] = std::move(w);
        }
        const auto t2 = now();
        L = waves[0].size();
        for (const auto& w : waves) PU_REQUIRE(w.size() == L, "pu_linksim_run: TX waveforms of one mode differ in length");
        noise_std.resize(static_cast<size_t>(m->n_snr) * pool);
        for (uint32_t i = 0; i < pool; ++i) {             // pu_channel_noise_std with the power sum taken once per waveform, not per SNR point
            const float acc = channel_power_sum(waves[i].data(), L);
            for (uint32_t si = 0; si < m->n_snr; ++si)
                noise_std[static_cast<size_t>(si) * pool + i] = channel_noise_std_from_sum(acc, L, m->snr_first_db + si * m->snr_step_db, convention);
        }
        if ((s = d_tx.reserve(static_cast<size_t>(pool) * L * sizeof(float))) != PU_OK) return s;
        if ((s = d_payload.reserve(payloads.size())) != PU_OK) return s;
        std::vector<float> flat(static_cast<size_t>(pool) * L);
        for (uint32_t i = 0; i < pool; ++i) std::copy(waves[i].begin(), waves[i].end(), flat.begin() + static_cast<size_t>(i) * L);
        PU_CUDA_TRY(cudaMemcpyAsync(d_tx.ptr, flat.data(), flat.size() * sizeof(float), cudaMemcpyHostToDevice, st));
        PU_CUDA_TRY(cudaMemcpyAsync(d_payload.ptr, payloads.data(), payloads.size(), cudaMemcpyHostToDevice, st));
        if (raw) {
            if ((s = d_coded.reserve(coded_pool.size())) != PU_OK) return s;
            PU_CUDA_TRY(cudaMemcpyAsync(d_coded.ptr, coded_pool.data(), coded_pool.size(), cudaMemcpyHostToDevice, st));
        }
        PU_CUDA_TRY(cudaStreamSynchronize(st));       // `flat` / `payloads` / `coded_pool` are pageable and go out of scope
        if (trace) fprintf(stderr, "[engine] mode %u: decoder %.3f s, demodulator %.3f s, TX pool %.3f s, noise levels + upload %.3f s\n", mode_index, secs(t0, t_ldpc),
                           secs(t_ldpc, t1), secs(t1, t2), secs(t2, now()));
        return PU_OK;
    }

    // fresh payloads: LDPC encode + modulate B payloads on the device into out[B][L] at column lead_samples + chirp_len (the caller clears
    // the rows when the mode has silence); B = 0 queries body_len.  Behind a chirp the peak normalisation waits for the pair (finish_rows).
    pu_status tx_batch(const uint8_t* d_pay, size_t B, float* out, size_t row, cudaStream_t st) {
        float* at = out ? out + md->lead_samples + chirp_len : nullptr;
        const float peak = chirp_len ? 0.0f : md->peak;
        const unsigned wf = md->waveform;
        if (frames) {
            size_t ncw = 0;
            return pu_frame_tx_batch(ofdm, ldpc, d_pay, pay_stride, frame_bytes, B, wf == PU_WF_OFDM_SC ? 1 : 0, peak, at, row, &body_len, &ncw,
                                     PU_MEM_DEVICE, st);
        }
        if (wf == PU_WF_OFDM || wf == PU_WF_OFDM_SC || wf == PU_WF_OFDM_CHIRP)
            return pu_ofdm_tx_batch(ofdm, ldpc, d_pay, kb, md->payload_bytes, B, wf == PU_WF_OFDM_SC ? 1 : 0, peak, at, row, &body_len, PU_MEM_DEVICE, st);
        if (wf == PU_WF_DPSK || wf == PU_WF_DPSK_ACQ)
            return pu_dpsk_tx_batch(dpsk, ldpc, d_pay, kb, md->payload_bytes, B, peak, at, row, &body_len, PU_MEM_DEVICE, st);
        return pu_mcdpsk_tx_batch(mcd, ldpc, d_pay, kb, md->payload_bytes, B, peak, at, row, &body_len, PU_MEM_DEVICE, st);
    }

    // fresh payloads, after tx_batch: the chirp pair and the peak normalisation, then the tools' CFO injector over the whole row
    pu_status finish_rows(float* out, size_t B, cudaStream_t st) {
        if (chirp_len) {
            chirp_peak_kernel<<<static_cast<unsigned>(B), 256, 0, st>>>(out, L, md->lead_samples, static_cast<const float*>(d_chirp.ptr), chirp_len,
                                                                       body_len, md->peak);
            ctx->launches.fetch_add(1);
            PU_CUDA_TRY(cudaGetLastError());
        }
        return tools_cfo ? pu_tools_cfo_apply_batch(tools_cfo, out, B, L, PU_MEM_DEVICE, st) : PU_OK;
    }

    // raw counts of the soft bits in llr (decoder order) against the coded bytes sent (Raw::coded row Raw::index[b]).  The acquiring
    // receivers' n_llr (NULL for the others) marks the soft bits they did not deliver as erasures.  It counts in the receiver's order, so
    // behind pu_llr_deinterleave_batch the counter finds the undelivered bits through the interleaver's permutation (its step).
    struct Raw {
        uint64_t* counters;                // [units of the batch][4]; NULL = no raw counts
        const uint8_t* coded;
        const uint32_t* index;
        const uint32_t* bin;
    };
    pu_status count_raw(const Raw& r, const float* llr, size_t B, const int32_t* n_llr, cudaStream_t st) {
        const size_t n = static_cast<size_t>(n_cw) * PU_LDPC_N;
        size_t step = 0;
        if (deinterleave) pu_channel_interleaver_perm(md->interleave_bps, PU_LDPC_N, nullptr, nullptr, &step);
        return count_raw_errors(ctx, llr, n, n, n_llr, r.coded, n / 8, r.index, r.bin, B, 10.0f, r.counters, st, static_cast<uint32_t>(step));
    }

    // fresh payloads with raw counts: the coded bytes of the batch's payload rows, before interleaving, as the transmitter encodes them
    pu_status encode_batch(const uint8_t* d_pay, size_t B, uint8_t* coded, cudaStream_t st) {
        const size_t stride = static_cast<size_t>(n_cw) * (PU_LDPC_N / 8);
        if (!frames) return pu_ldpc_encode_batch(ldpc, d_pay, kb, md->payload_bytes, B, coded, stride, PU_MEM_DEVICE, st);
        size_t ncw = 0;
        return pu_frame_encode_batch(ldpc, d_pay, pay_stride, frame_bytes, B, coded, stride, &ncw, PU_MEM_DEVICE, st);
    }

    // frame modes: demodulate every codeword of the frame (llr [B][n_cw * 648]) -> decodeFrame (cw_* [B * n_cw] codeword scratch) ->
    // frame_out [B][frame_bytes], frame_len [B], info [B][5]; ncw [B] = codewords the acquiring receivers delivered
    pu_status receive_frames(const float* rx, size_t B, float* llr, int32_t* n_llr, int32_t* sync_i, float* sync_f, uint8_t* cw_bytes, uint8_t* cw_ok,
                             int32_t* cw_iters, uint8_t* frame_out, int32_t* frame_len, int32_t* info, int32_t* ncw, const Raw& raw, cudaStream_t st) {
        pu_status s = PU_OK;
        const size_t stride = static_cast<size_t>(n_cw) * PU_LDPC_N;
        const unsigned wf = md->waveform;
        if (wf == PU_WF_OFDM) {
            if ((s = pu_ofdm_presynced_batch(ofdm, rx, B, L, 2, nullptr, nullptr, llr, stride, nullptr, nullptr, PU_MEM_DEVICE, st)) != PU_OK) return s;
            ncw = nullptr;
            n_llr = nullptr;
        } else {
            PU_CUDA_TRY(cudaMemsetAsync(llr, 0, B * stride * sizeof(float), st));
            if (wf == PU_WF_OFDM_SC)
                s = pu_ofdm_process_batch(ofdm, rx, B, L, md->chunk ? md->chunk : 960, 0.0f, llr, stride, n_llr, sync_i, sync_f, nullptr, PU_MEM_DEVICE, st);
            else
                s = pu_ofdm_chirp_receive_batch(ofdm, rx, B, L, 0.0f, llr, stride, n_llr, sync_i, sync_f, nullptr, PU_MEM_DEVICE, st);
            if (s != PU_OK) return s;
            frame_codewords_kernel<<<static_cast<unsigned>((B + 255) / 256), 256, 0, st>>>(ncw, n_llr, static_cast<int>(n_cw), B);
            ctx->launches.fetch_add(1);
            PU_CUDA_TRY(cudaGetLastError());
        }
        if (deinterleave && (s = llr_deinterleave_enqueue(ctx, llr, B, stride, n_cw, md->interleave_bps, st)) != PU_OK) return s;
        if (raw.counters && (s = count_raw(raw, llr, B, n_llr, st)) != PU_OK) return s;
        return frame_decode_enqueue(ctx, ldpc, llr, B, static_cast<int>(n_cw), ncw, cw_bytes, cw_ok, cw_iters, frame_out, frame_bytes, frame_len, info, st);
    }

    // demodulate -> decode (device pointers, stream st); scratch: llr [B][648], n_llr [B], sync [B][8] (int/float)
    pu_status receive(const float* rx, size_t B, float* llr, int32_t* n_llr, int32_t* sync_i, float* sync_f, uint8_t* info, uint8_t* ok, int32_t* iters,
                      const Raw& raw, cudaStream_t st) {
        pu_status s = PU_OK;
        bool mask = false;
        const unsigned wf = md->waveform;
        if (wf == PU_WF_OFDM && !raw.counters)
            return pu_receive_decode_batch(ofdm, ldpc, rx, B, L, 2, nullptr, nullptr, info, kb, ok, iters, PU_MEM_DEVICE, st);
        if (wf == PU_WF_OFDM) {          // the two halves of pu_receive_decode_batch's device path, with the soft bits counted in between
            const int n_sym = static_cast<int>(L / static_cast<size_t>(pu_ofdm_symbol_samples(ofdm)));
            if (static_cast<size_t>(std::max(0, n_sym - 2)) * static_cast<size_t>(pu_ofdm_bits_per_symbol(ofdm)) < PU_LDPC_N)
                PU_CUDA_TRY(cudaMemsetAsync(llr, 0, B * PU_LDPC_N * sizeof(float), st));   // frames shorter than a codeword: erasures
            if ((s = pu_ofdm_presynced_batch(ofdm, rx, B, L, 2, nullptr, nullptr, llr, PU_LDPC_N, nullptr, nullptr, PU_MEM_DEVICE, st)) != PU_OK) return s;
            if ((s = count_raw(raw, llr, B, nullptr, st)) != PU_OK) return s;
            return pu_ldpc_decode_batch(ldpc, llr, PU_LDPC_N, B, info, kb, ok, iters, PU_MEM_DEVICE, st);
        }
        if (wf != PU_WF_DPSK && wf != PU_WF_MCDPSK) PU_CUDA_TRY(cudaMemsetAsync(llr, 0, B * PU_LDPC_N * sizeof(float), st));
        switch (wf) {
            case PU_WF_OFDM_SC:
                s = pu_ofdm_process_batch(ofdm, rx, B, L, md->chunk ? md->chunk : 960, 0.0f, llr, PU_LDPC_N, n_llr, sync_i, sync_f, nullptr, PU_MEM_DEVICE, st);
                mask = true; break;
            case PU_WF_OFDM_CHIRP:
                s = pu_ofdm_chirp_receive_batch(ofdm, rx, B, L, 0.0f, llr, PU_LDPC_N, n_llr, sync_i, sync_f, nullptr, PU_MEM_DEVICE, st);
                mask = true; break;
            case PU_WF_DPSK:
                s = pu_dpsk_demod_soft_batch(dpsk, rx, B, L, 39u * md->dpsk.samples_per_symbol, 1, nullptr, nullptr, llr, PU_LDPC_N, PU_MEM_DEVICE, st);
                break;
            case PU_WF_DPSK_ACQ:
                s = pu_dpsk_receive_batch(dpsk, rx, B, L, llr, PU_LDPC_N, n_llr, sync_i, sync_f, sync_f + B, PU_MEM_DEVICE, st);
                mask = true; break;
            case PU_WF_MCDPSK:
                s = pu_mcdpsk_demod_soft_batch(mcd, rx, B, L, llr, PU_LDPC_N, nullptr, PU_MEM_DEVICE, st);
                break;
            default:
                s = pu_mcdpsk_chirp_receive_batch(mcd, rx, B, L, 0.0f, llr, PU_LDPC_N, n_llr, sync_i, sync_f, sync_f + 4 * B, PU_MEM_DEVICE, st);
                mask = true; break;
        }
        if (s != PU_OK) return s;
        if (deinterleave && (s = llr_deinterleave_enqueue(ctx, llr, B, PU_LDPC_N, 1, md->interleave_bps, st)) != PU_OK) return s;
        if (raw.counters && (s = count_raw(raw, llr, B, mask ? n_llr : nullptr, st)) != PU_OK) return s;
        if ((s = pu_ldpc_decode_batch(ldpc, llr, PU_LDPC_N, B, info, kb, ok, iters, PU_MEM_DEVICE, st)) != PU_OK) return s;
        if (mask) {
            mask_short_kernel<<<static_cast<unsigned>((B + 255) / 256), 256, 0, st>>>(ok, n_llr, B);
            ctx->launches.fetch_add(1);
            PU_CUDA_TRY(cudaGetLastError());
        }
        return PU_OK;
    }
};

// ---- manifest: one text line per finished unit, in a per-rank shard file ----------------------------------------------------------
struct Manifest {
    std::string dir;
    FILE* f = nullptr;
    ~Manifest() { if (f) fclose(f); }

    // reads every shard of `dir`; returns false on a key mismatch
    // nc = counters per record: 6, or 10 in a raw run (the 6, then the 4 raw counters)
    bool load(const std::string& d, uint64_t key, uint64_t run_id, uint64_t n_units, int nc, std::vector<uint8_t>& done,
              std::vector<uint64_t>& rec /* [n_units][nc] */) {
        dir = d;
        char own[64];
        snprintf(own, sizeof own, "shard-%016llx-", static_cast<unsigned long long>(run_id));
        mkdir(dir.c_str(), 0777);
        DIR* dp = opendir(dir.c_str());
        if (!dp) return true;
        bool ok = true;
        while (dirent* e = readdir(dp)) {
            const std::string name = e->d_name;
            if (name.rfind("shard-", 0) != 0) continue;
            if (name.rfind(own, 0) == 0) continue;       // written by this launch (this rank earlier, or a peer that started first)
            FILE* in = fopen((dir + "/" + name).c_str(), "r");
            if (!in) continue;
            char line[256];
            while (fgets(line, sizeof line, in)) {
                unsigned long long k = 0, u = 0, c[10];
                if (line[0] == '#') {
                    if (sscanf(line, "# key %llx", &k) == 1 && k != key) ok = false;
                    continue;
                }
                // a torn last line (killed while appending) does not parse to 1 + nc fields + the end mark and is ignored
                char endmark = 0;
                const int got = nc == 6 ? sscanf(line, "%llu %llu %llu %llu %llu %llu %llu %c", &u, &c[0], &c[1], &c[2], &c[3], &c[4], &c[5], &endmark)
                                        : sscanf(line, "%llu %llu %llu %llu %llu %llu %llu %llu %llu %llu %llu %c", &u, &c[0], &c[1], &c[2], &c[3], &c[4],
                                                 &c[5], &c[6], &c[7], &c[8], &c[9], &endmark);
                if (got != nc + 2 || endmark != ';') continue;
                if (u >= n_units || done[u]) continue;
                done[u] = 1;
                for (int i = 0; i < nc; ++i) rec[u * nc + i] = c[i];
            }
            fclose(in);
        }
        closedir(dp);
        return ok;
    }
    bool open_shard(uint64_t key, uint64_t run_id, uint32_t rank, uint32_t world) {
        char name[128];
        snprintf(name, sizeof name, "/shard-%016llx-r%uof%u.txt", static_cast<unsigned long long>(run_id), rank, world);
        f = fopen((dir + name).c_str(), "a");
        if (!f) return false;
        fprintf(f, "# key %llx\n", static_cast<unsigned long long>(key));
        fflush(f);
        return true;
    }
    void append(uint64_t unit, const uint64_t* c, const uint64_t* raw /* NULL in a plain run */) {
        if (!f) return;
        fprintf(f, "%llu %llu %llu %llu %llu %llu %llu", (unsigned long long)unit, (unsigned long long)c[0], (unsigned long long)c[1],
                (unsigned long long)c[2], (unsigned long long)c[3], (unsigned long long)c[4], (unsigned long long)c[5]);
        if (raw) fprintf(f, " %llu %llu %llu %llu", (unsigned long long)raw[0], (unsigned long long)raw[1], (unsigned long long)raw[2], (unsigned long long)raw[3]);
        fprintf(f, " ;\n");
    }
    void flush() { if (f) fflush(f); }
};

struct Slot {       // one batch in flight; the buffers live in the context (grow-only, reused across calls)
    Buffer *h_desc = nullptr, *d_desc = nullptr, *d_cnt = nullptr, *h_cnt = nullptr;
    cudaEvent_t ev = nullptr;
    std::vector<uint64_t> units;       // unit ids of the batch, bin order
    uint32_t mode = 0;
    size_t frames = 0;
    bool busy = false;
};

void partition(const pu_sweep_desc* d, const SweepPlan& p, const uint8_t* done, uint32_t* owner, double* cost_out, std::vector<double>* load_out) {
    const uint64_t n = p.unit0.back();
    std::vector<double> cost(n);
    std::vector<uint64_t> order;
    order.reserve(n);
    for (uint64_t u = 0; u < n; ++u) {
        uint32_t m, s, nt; uint64_t t0;
        unit_decode(d, p, u, &m, &s, &t0, &nt);
        cost[u] = unit_cost(p, d->modes[m], m, s, nt);
        owner[u] = kNoOwner;
        if (!(done && done[u])) order.push_back(u);
    }
    std::stable_sort(order.begin(), order.end(), [&](uint64_t a, uint64_t b) { return cost[a] > cost[b]; });
    // longest processing time first: every unit goes to the least loaded rank (ties: lowest rank)
    using Item = std::pair<double, uint32_t>;
    std::priority_queue<Item, std::vector<Item>, std::greater<Item>> heap;
    for (uint32_t r = 0; r < d->world; ++r) heap.push({0.0, r});
    std::vector<double> load(d->world, 0.0);
    for (uint64_t u : order) {
        Item it = heap.top();
        heap.pop();
        owner[u] = it.second;
        it.first += cost[u];
        load[it.second] = it.first;
        heap.push(it);
    }
    if (cost_out) std::copy(cost.begin(), cost.end(), cost_out);
    if (load_out) *load_out = load;
}

}  // namespace
}  // namespace pu

extern "C" {

pu_status pu_channel_preset(int preset, pu_channel_config* out) {
    PU_REQUIRE(out, "pu_channel_preset: out is NULL");
    // ccir:: (src/sim/hf_channel.hpp:305-381) and itu_r_f1487:: (:402-487) carry the same numbers per condition
    static const float table[5][4] = {{0.0f, 0.0f, 1.0f, 0.0f}, {0.5f, 0.1f, 0.707f, 0.707f}, {1.0f, 0.5f, 0.707f, 0.707f},
                                      {2.0f, 1.0f, 0.707f, 0.707f}, {0.5f, 10.0f, 0.707f, 0.707f}};
    PU_REQUIRE(preset >= PU_CH_AWGN && preset <= PU_CH_ITU_FLUTTER, "pu_channel_preset: unknown preset");
    const int row = preset <= PU_CH_FLUTTER ? preset : preset - 4;
    const bool fading = row != 0;
    *out = pu_channel_config{table[row][0], table[row][1], table[row][2], table[row][3], 48000u, fading ? 1u : 0u, fading ? 1u : 0u, 1u};
    return PU_OK;
}

uint64_t pu_sweep_unit_count(const pu_sweep_desc* d) {
    pu::SweepPlan p;
    return pu::make_plan(d, &p) ? p.unit0.back() : 0;
}
uint32_t pu_sweep_point_count(const pu_sweep_desc* d) {
    pu::SweepPlan p;
    return pu::make_plan(d, &p) ? p.point0.back() : 0;
}

pu_status pu_sweep_partition(const pu_sweep_desc* d, const uint8_t* done, uint32_t* owner, double* cost) {
    pu::SweepPlan p;
    PU_REQUIRE(pu::make_plan(d, &p) && owner, "pu_sweep_partition: invalid sweep description");
    pu::partition(d, p, done, owner, cost, nullptr);
    return PU_OK;
}

pu_status pu_sweep_unit(const pu_sweep_desc* d, uint64_t u, uint32_t* mode, uint32_t* snr_index, uint64_t* first_trial, uint32_t* n_trials) {
    pu::SweepPlan p;
    PU_REQUIRE(pu::make_plan(d, &p) && u < p.unit0.back(), "pu_sweep_unit: invalid sweep description or unit");
    uint32_t m, s, nt; uint64_t t0;
    pu::unit_decode(d, p, u, &m, &s, &t0, &nt);
    if (mode) *mode = m;
    if (snr_index) *snr_index = s;
    if (first_trial) *first_trial = t0;
    if (n_trials) *n_trials = nt;
    return PU_OK;
}

void pu_sweep_payload(uint64_t base_seed, uint32_t mode, uint32_t index, uint8_t* out, size_t n_bytes) {
    uint64_t x = (base_seed ? base_seed : 0xB200) * 0x9e3779b97f4a7c15ull ^ (static_cast<uint64_t>(mode) << 32) ^ index;
    for (size_t i = 0; i < n_bytes; i += 8) {
        const uint64_t v = pu::splitmix64(x);
        for (size_t j = 0; j < 8 && i + j < n_bytes; ++j) out[i + j] = static_cast<uint8_t>(v >> (8 * j));
    }
}

void pu_wilson_interval(uint64_t errors, uint64_t n, double z, double* lo, double* hi) {
    double a = 0.0, b = 1.0;
    if (n > 0) {
        const double p = static_cast<double>(errors) / n, den = 1.0 + z * z / n;
        const double mid = (p + z * z / (2.0 * n)) / den;
        const double half = z * std::sqrt(p * (1.0 - p) / n + z * z / (4.0 * static_cast<double>(n) * n)) / den;
        a = std::max(0.0, mid - half);
        b = std::min(1.0, mid + half);
    }
    if (lo) *lo = a;
    if (hi) *hi = b;
}

pu_status pu_linksim_run(pu_ctx* ctx, const pu_sweep_desc* d, uint64_t* counters, pu_sweep_stats* stats) {
    return pu_linksim_run_raw(ctx, d, counters, nullptr, stats);
}

pu_status pu_linksim_run_raw(pu_ctx* ctx, const pu_sweep_desc* d, uint64_t* counters, uint64_t* raw, pu_sweep_stats* stats) {
    PU_REQUIRE(ctx && d && counters, "pu_linksim_run: NULL argument");
    pu::SweepPlan p;
    PU_REQUIRE(pu::make_plan(d, &p), "pu_linksim_run: invalid sweep description");
    PU_CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const uint64_t n_units = p.unit0.back();
    const uint32_t n_points = p.point0.back();
    std::fill(counters, counters + static_cast<size_t>(n_points) * 6, uint64_t(0));
    if (raw) std::fill(raw, raw + static_cast<size_t>(n_points) * 4, uint64_t(0));
    const int nc = raw ? 10 : 6;          // counters per unit: the 6, then the 4 raw counters of a raw run
    pu_sweep_stats stt{};
    stt.units_total = n_units;

    // ---- resume
    std::vector<uint8_t> done(n_units, 0);
    std::vector<uint64_t> rec;
    pu::Manifest man;
    const uint64_t key = pu::desc_key(d, p, raw != nullptr);
    if (d->manifest_dir && d->manifest_dir[0]) {
        rec.assign(n_units * nc, 0);
        if (!man.load(d->manifest_dir, key, d->run_id, n_units, nc, done, rec)) {
            pu::set_error("pu_linksim_run: %s holds the manifest of a different sweep (key mismatch); use an empty directory", d->manifest_dir);
            return PU_ERR_INVALID;
        }
        if (!man.open_shard(key, d->run_id, d->rank, d->world)) {
            pu::set_error("pu_linksim_run: cannot write a shard file in %s", d->manifest_dir);
            return PU_ERR_INVALID;
        }
        for (uint64_t u = 0; u < n_units; ++u) {
            if (!done[u]) continue;
            ++stt.units_resumed;
            if (d->rank != 0) continue;        // resumed counters enter the job total once
            uint32_t m, s, nt; uint64_t t0;
            pu::unit_decode(d, p, u, &m, &s, &t0, &nt);
            for (int i = 0; i < 6; ++i) counters[(p.point0[m] + s) * 6 + i] += rec[u * nc + i];
            if (raw)
                for (int i = 0; i < 4; ++i) raw[(p.point0[m] + s) * 4 + i] += rec[u * nc + 6 + i];
        }
    }
    std::vector<uint32_t> owner(n_units);
    std::vector<double> cost(n_units), load;
    pu::partition(d, p, done.data(), owner.data(), cost.data(), &load);
    stt.busy_cost = load[d->rank];
    stt.total_cost = std::accumulate(load.begin(), load.end(), 0.0);

    // ---- batches in flight
    pu::Slot slots[2];
    pu::Buffer &d_rx = ctx->sweep[0], &d_llr = ctx->sweep[1], &d_info = ctx->sweep[2], &d_ok = ctx->sweep[3], &d_iters = ctx->sweep[4],
               &d_nllr = ctx->sweep[5], &d_sync = ctx->sweep[6], &d_ftx = ctx->sweep[15], &d_fpay = ctx->sweep[16], &d_fstd = ctx->sweep[17],
               &d_fout = ctx->sweep[18], &d_finfo = ctx->sweep[19], &d_fcoded = ctx->sweep[20];
    for (int i = 0; i < 2; ++i) {
        pu::Slot& sl = slots[i];
        sl.h_desc = &ctx->sweep[7 + 4 * i]; sl.d_desc = &ctx->sweep[8 + 4 * i]; sl.d_cnt = &ctx->sweep[9 + 4 * i]; sl.h_cnt = &ctx->sweep[10 + 4 * i];
        sl.h_desc->pinned_host = true;
        sl.h_cnt->pinned_host = true;
        if (!ctx->sweep_ev[i] && cudaEventCreateWithFlags(&ctx->sweep_ev[i], cudaEventDisableTiming) != cudaSuccess) {
            ctx->sweep_ev[i] = nullptr;
            pu::set_error("pu_linksim_run: cudaEventCreate failed");
            return PU_ERR_CUDA;
        }
        sl.ev = ctx->sweep_ev[i];
    }
    auto cleanup = [&]() {};
    auto harvest = [&](pu::Slot& sl) -> pu_status {
        if (!sl.busy) return PU_OK;
        const auto t_wait = std::chrono::steady_clock::now();
        PU_CUDA_TRY(cudaEventSynchronize(sl.ev));
        stt.wait_seconds += std::chrono::duration<double>(std::chrono::steady_clock::now() - t_wait).count();
        const uint64_t* hc = static_cast<const uint64_t*>(sl.h_cnt->ptr);
        const uint64_t* hr = hc + sl.units.size() * 6;      // raw counters [units][4] behind the [units][6]
        for (size_t i = 0; i < sl.units.size(); ++i) {
            uint32_t m, s, nt; uint64_t t0;
            pu::unit_decode(d, p, sl.units[i], &m, &s, &t0, &nt);
            for (int k = 0; k < 6; ++k) counters[(p.point0[m] + s) * 6 + k] += hc[i * 6 + k];
            if (raw)
                for (int k = 0; k < 4; ++k) raw[(p.point0[m] + s) * 4 + k] += hr[i * 4 + k];
            man.append(sl.units[i], hc + i * 6, raw ? hr + i * 4 : nullptr);
        }
        man.flush();
        stt.units_run += sl.units.size();
        stt.frames_run += sl.frames;
        sl.busy = false;
        return PU_OK;
    };

    const auto t_begin = std::chrono::steady_clock::now();
    pu_status rs = PU_OK;
    pu_ldpc* decoders[8] = {};
    uint64_t budget = d->max_units ? d->max_units : ~uint64_t(0);
    int k = 0;
    for (uint32_t m = 0; m < d->n_modes && rs == PU_OK && budget > 0; ++m) {
        std::vector<uint64_t> mine;
        for (uint64_t u = p.unit0[m]; u < p.unit0[m + 1]; ++u)
            if (owner[u] == d->rank) mine.push_back(u);
        if (mine.empty()) continue;
        pu::ModeEngine eng;
        const auto t_setup = std::chrono::steady_clock::now();
        const unsigned rate = d->modes[m].code_rate;      // one decoder per code rate for the whole run (its tables take longer to build than a mode's)
        if (rate < 8 && !decoders[rate] && (rs = pu_ldpc_create(ctx, static_cast<int>(rate), static_cast<int>(p.max_iter), &decoders[rate])) != PU_OK) break;
        if ((rs = eng.build(ctx, &d->modes[m], m, p, st, rate < 8 ? decoders[rate] : nullptr, raw != nullptr)) != PU_OK) break;
        const double t_build = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_setup).count();
        stt.setup_seconds += t_build;
        if (std::getenv("PU_SWEEP_TRACE"))
            fprintf(stderr, "[pu_linksim_run] rank %u mode %u waveform %u: engine set-up %.3f s (%zu samples per frame, pool %u)\n", d->rank, m,
                    d->modes[m].waveform, t_build, eng.L, eng.pool);
        const size_t L = eng.L, kb = eng.kb, ncw = eng.n_cw;
        // (fresh payloads keep the clean TX batch next to the received one: half as many frames per batch; frame modes count their soft bits)
        const size_t bytes_per_trial = L * sizeof(float) * (eng.fresh ? 2 : 1) + (eng.frames ? ncw * PU_LDPC_N * sizeof(float) : 0);
        const size_t max_frames = std::max<size_t>(1, std::min<uint64_t>(p.batch_bytes / bytes_per_trial, (uint64_t(1) << 22)));
        const size_t cap = std::max<size_t>(max_frames, p.block);      // a unit is never split: the smallest batch is one unit
        if ((rs = d_rx.reserve(cap * L * sizeof(float))) != PU_OK || (rs = d_llr.reserve(cap * ncw * PU_LDPC_N * sizeof(float))) != PU_OK ||
            (rs = d_info.reserve(cap * ncw * kb)) != PU_OK || (rs = d_ok.reserve(cap * ncw)) != PU_OK || (rs = d_iters.reserve(cap * ncw * 4)) != PU_OK ||
            (rs = d_nllr.reserve(cap * 4)) != PU_OK || (rs = d_sync.reserve(cap * 12 * 4)) != PU_OK)
            break;
        if (eng.fresh && ((rs = d_ftx.reserve(cap * L * sizeof(float))) != PU_OK || (rs = d_fpay.reserve(cap * eng.pay_stride)) != PU_OK ||
                          (rs = d_fstd.reserve(cap * sizeof(float))) != PU_OK))
            break;
        if (eng.fresh && raw && (rs = d_fcoded.reserve(cap * ncw * (PU_LDPC_N / 8))) != PU_OK) break;
        // frame modes: reassembled frames; frame_len [cap], info [cap][5], codewords delivered [cap]
        if (eng.frames && ((rs = d_fout.reserve(cap * eng.frame_bytes)) != PU_OK || (rs = d_finfo.reserve(cap * 7 * sizeof(int32_t))) != PU_OK))
            break;
        size_t next = 0;
        while (next < mine.size() && budget > 0 && rs == PU_OK) {
            pu::Slot& sl = slots[k & 1];
            ++k;
            if ((rs = harvest(sl)) != PU_OK) break;
            // ---- the batch: as many of this rank's units of the mode as fit
            sl.units.clear();
            sl.mode = m;
            size_t B = 0;
            while (next < mine.size() && budget > 0) {
                uint32_t mm, s, nt; uint64_t t0;
                pu::unit_decode(d, p, mine[next], &mm, &s, &t0, &nt);
                if (!sl.units.empty() && B + nt > cap) break;
                sl.units.push_back(mine[next++]);
                B += nt;
                --budget;
            }
            sl.frames = B;
            const size_t nu = sl.units.size();
            // descriptors: tx_index u32 | noise_std f32 | bin u32 | seed u64 (8-byte aligned at the end)
            const size_t off_std = B * 4, off_bin = B * 8, off_seed = ((B * 12 + 7) / 8) * 8, desc_bytes = off_seed + B * 8;
            if ((rs = sl.h_desc->reserve(desc_bytes)) != PU_OK || (rs = sl.d_desc->reserve(desc_bytes)) != PU_OK ||
                (rs = sl.d_cnt->reserve(nu * nc * 8)) != PU_OK || (rs = sl.h_cnt->reserve(nu * nc * 8)) != PU_OK)
                break;
            unsigned char* hd = static_cast<unsigned char*>(sl.h_desc->ptr);
            uint32_t* h_tx = reinterpret_cast<uint32_t*>(hd);
            float* h_std = reinterpret_cast<float*>(hd + off_std);
            uint32_t* h_bin = reinterpret_cast<uint32_t*>(hd + off_bin);
            uint64_t* h_seed = reinterpret_cast<uint64_t*>(hd + off_seed);
            size_t at = 0;
            const auto t_fill = std::chrono::steady_clock::now();
            for (size_t i = 0; i < nu; ++i) {
                uint32_t mm, s, nt; uint64_t t0;
                pu::unit_decode(d, p, sl.units[i], &mm, &s, &t0, &nt);
                const uint64_t hi = (p.base_seed << 40) ^ (static_cast<uint64_t>(m) << 56) ^ (static_cast<uint64_t>(s) << 32);
                const float* stdrow = eng.fresh ? nullptr : eng.noise_std.data() + static_cast<size_t>(s) * eng.pool;
                for (uint32_t j = 0; j < nt; ++j, ++at) {
                    const uint64_t trial = t0 + j;
                    if (eng.fresh) {             // the batch is its own pool; the "std" column carries the SNR factor of pu_channel_noise_std_batch
                        h_tx[at] = static_cast<uint32_t>(at); h_std[at] = eng.noise_std[s];
                    } else {
                        const uint32_t tx = static_cast<uint32_t>(trial % eng.pool);
                        h_tx[at] = tx; h_std[at] = stdrow[tx];
                    }
                    h_bin[at] = static_cast<uint32_t>(i); h_seed[at] = hi ^ trial;
                }
            }
            stt.fill_seconds += std::chrono::duration<double>(std::chrono::steady_clock::now() - t_fill).count();
            unsigned char* dd = static_cast<unsigned char*>(sl.d_desc->ptr);
            auto launch = [&]() -> pu_status {
                PU_CUDA_TRY(cudaMemcpyAsync(dd, hd, desc_bytes, cudaMemcpyHostToDevice, st));
                PU_CUDA_TRY(cudaMemsetAsync(sl.d_cnt->ptr, 0, nu * nc * 8, st));
                float* rx = static_cast<float*>(d_rx.ptr);
                const float* tx_pool = static_cast<const float*>(eng.d_tx.ptr);
                const float* stds = reinterpret_cast<const float*>(dd + off_std);
                const uint8_t* payloads = static_cast<const uint8_t*>(eng.d_payload.ptr);
                const uint8_t* coded = static_cast<const uint8_t*>(eng.d_coded.ptr);
                size_t pool_count = eng.pool;
                pu_status s2;
                if (eng.fresh) {                 // payload -> encode -> modulate for every frame of the batch, then its own noise level
                    uint8_t* pay = static_cast<uint8_t*>(d_fpay.ptr);
                    float* ftx = static_cast<float*>(d_ftx.ptr);
                    const uint64_t* seeds = reinterpret_cast<const uint64_t*>(dd + off_seed);
                    if (eng.frames) {
                        pu::fresh_frame_kernel<<<static_cast<unsigned>((B + 7) / 8), 256, 0, st>>>(pay, eng.pay_stride, d->modes[m].frame_payload_bytes,
                                                                                                   static_cast<int>(d->modes[m].code_rate), seeds, B);
                    } else {
                        const size_t words = B * ((kb + 7) / 8);
                        pu::fresh_payload_kernel<<<static_cast<unsigned>((words + 255) / 256), 256, 0, st>>>(pay, kb, d->modes[m].payload_bytes, seeds, B);
                    }
                    ctx->launches.fetch_add(1);
                    PU_CUDA_TRY(cudaGetLastError());
                    if (raw && (s2 = eng.encode_batch(pay, B, static_cast<uint8_t*>(d_fcoded.ptr), st)) != PU_OK) return s2;
                    if (raw) coded = static_cast<const uint8_t*>(d_fcoded.ptr);
                    if (d->modes[m].lead_samples || d->modes[m].tail_samples) PU_CUDA_TRY(cudaMemsetAsync(ftx, 0, B * L * sizeof(float), st));
                    if ((s2 = eng.tx_batch(pay, B, ftx, L, st)) != PU_OK) return s2;
                    if ((s2 = eng.finish_rows(ftx, B, st)) != PU_OK) return s2;
                    if ((s2 = pu_channel_noise_std_batch(ctx, ftx, L, L, B, stds, eng.convention, static_cast<float*>(d_fstd.ptr), st)) != PU_OK) return s2;
                    tx_pool = ftx; stds = static_cast<const float*>(d_fstd.ptr); payloads = pay; pool_count = B;
                }
                s2 = pu_channel_apply_batch(ctx, &eng.ch, tx_pool, L, pool_count, reinterpret_cast<const uint32_t*>(dd), stds,
                                            reinterpret_cast<const uint64_t*>(dd + off_seed), B, L, rx, PU_MEM_DEVICE, st);
                if (s2 != PU_OK) return s2;
                uint8_t* info = static_cast<uint8_t*>(d_info.ptr);
                uint8_t* ok = static_cast<uint8_t*>(d_ok.ptr);
                int32_t* iters = static_cast<int32_t*>(d_iters.ptr);
                const uint32_t* tx_index = reinterpret_cast<const uint32_t*>(dd);
                const uint32_t* bins = reinterpret_cast<const uint32_t*>(dd + off_bin);
                uint64_t* cnt = static_cast<uint64_t*>(sl.d_cnt->ptr);
                const pu::ModeEngine::Raw rw{raw ? cnt + nu * 6 : nullptr, coded, tx_index, bins};
                if (eng.frames) {
                    uint8_t* fout = static_cast<uint8_t*>(d_fout.ptr);
                    int32_t* flen = static_cast<int32_t*>(d_finfo.ptr);
                    int32_t* finfo = flen + cap;
                    s2 = eng.receive_frames(rx, B, static_cast<float*>(d_llr.ptr), static_cast<int32_t*>(d_nllr.ptr), static_cast<int32_t*>(d_sync.ptr),
                                            reinterpret_cast<float*>(static_cast<int32_t*>(d_sync.ptr) + 4 * cap), info, ok, iters, fout, flen, finfo,
                                            finfo + 5 * cap, rw, st);
                    if (s2 != PU_OK) return s2;
                    s2 = pu::count_frame_errors(ctx, fout, eng.frame_bytes, flen, finfo, payloads, eng.pay_stride, tx_index, bins, eng.frame_bytes,
                                                static_cast<int>(ncw), B, cnt, st);
                } else {
                    s2 = eng.receive(rx, B, static_cast<float*>(d_llr.ptr), static_cast<int32_t*>(d_nllr.ptr), static_cast<int32_t*>(d_sync.ptr),
                                     reinterpret_cast<float*>(static_cast<int32_t*>(d_sync.ptr) + 4 * cap), info, ok, iters, rw, st);
                    if (s2 != PU_OK) return s2;
                    s2 = pu_count_errors(ctx, info, kb, ok, iters, payloads, kb, tx_index, bins, d->modes[m].payload_bytes, B, cnt, st);
                }
                if (s2 != PU_OK) return s2;
                PU_CUDA_TRY(cudaMemcpyAsync(sl.h_cnt->ptr, sl.d_cnt->ptr, nu * nc * 8, cudaMemcpyDeviceToHost, st));
                PU_CUDA_TRY(cudaEventRecord(sl.ev, st));
                return PU_OK;
            };
            const auto t_enq = std::chrono::steady_clock::now();
            if ((rs = launch()) != PU_OK) break;
            stt.enqueue_seconds += std::chrono::duration<double>(std::chrono::steady_clock::now() - t_enq).count();
            sl.busy = true;
        }
        // the engine's device buffers go away with it: drain both slots before leaving the mode
        for (auto& sl : slots) { const pu_status hs = harvest(sl); if (rs == PU_OK) rs = hs; }
    }
    if (rs != PU_OK) (void)cudaStreamSynchronize(st);
    for (pu_ldpc* h : decoders) if (h) pu_ldpc_destroy(h);
    for (auto& sl : slots) sl.busy = false;
    stt.seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_begin).count();
    cleanup();
    if (stats) *stats = stt;
    return rs;
}

pu_status pu_counters_allreduce(pu_ctx* ctx, uint64_t* counters, size_t n, void* nccl_comm, pu_memspace space, void* stream) {
    PU_REQUIRE(ctx && (counters || n == 0), "pu_counters_allreduce: NULL argument");
    if (!nccl_comm || n == 0) return PU_OK;
    // ncclResult_t ncclAllReduce(const void* sendbuff, void* recvbuff, size_t count, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t)
    using AllReduce = int (*)(const void*, void*, size_t, int, int, void*, cudaStream_t);
    static AllReduce fn = [] {
        void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);      // the copy the host process already loaded (torch's), if any
        if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        return h ? reinterpret_cast<AllReduce>(dlsym(h, "ncclAllReduce")) : nullptr;
    }();
    if (!fn) {
        pu::set_error("pu_counters_allreduce: libnccl.so.2 not found (dlopen): %s", dlerror());
        return PU_ERR_UNSUPPORTED;
    }
    PU_CUDA_TRY(cudaSetDevice(ctx->device));
    cudaStream_t st = pu::pick_stream(ctx, stream, space);
    constexpr int kNcclUint64 = 5, kNcclSum = 0;
    auto allreduce = [&](uint64_t* dbuf) -> pu_status {
        const int r = fn(dbuf, dbuf, n, kNcclUint64, kNcclSum, nccl_comm, st);
        if (r != 0) {
            pu::set_error("pu_counters_allreduce: ncclAllReduce failed with ncclResult_t %d", r);
            return PU_ERR_CUDA;
        }
        return PU_OK;
    };
    if (space == PU_MEM_DEVICE) return allreduce(counters);
    pu::HostStage hs(ctx, st, 1);
    uint64_t* dbuf;
    hs.inout(&dbuf, counters, n);
    return hs.run([&](size_t) { return allreduce(dbuf); });
}

}  // extern "C"
