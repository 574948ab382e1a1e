// tools/pu_sweep.cpp — C++20 host program of the config-5 sweep (BASELINE.json: "full adaptive-mode FER/BER waterfall (all waveforms
// x rates x SNR points x seeds) sharded across 8 x B200"): one process per GPU, everything heavy behind the C ABI of
// include/pu/pu_capi.h (pu_linksim_run), NCCL only to sum the counter tables.  The reference's shape: the per-(waveform, channel,
// SNR, CFO) matrix of tests/regression_matrix.sh:139-243 over the trial loop of tools/test_iwaveform.cpp:597-806.
//
//   torchrun-style launch (RANK / WORLD_SIZE / LOCAL_RANK in the environment), or a single process:
//     projectultra_b200/pu_sweep --table reduced --trials 16384 [--block 2048] [--manifest DIR] [--out rows.jsonl] [--fresh] [--frame-bytes N]
//                                [--interleave] [--raw]
//   tables: smoke (4 modes, seconds), reduced (one mode per waveform family and channel + the chirp-acquired CFO rows of the regression matrix), config5 (105 modes x 40 SNR points),
//   frames (whole-frame FER of protocol-v2 DATA frames of 200 and 1000 payload bytes, or N with --frame-bytes, over AWGN / good / poor)
//   --interleave: every OFDM and MC-DPSK codeword through ChannelInterleaver(bits per symbol, 648) as the reference's IWaveform path
//   does (OFDM: data carriers x bits per carrier = ChannelInterleaver(60) for the M1 DQPSK modes; MC-DPSK: carriers x bits per carrier);
//   single-carrier DPSK rows stay without
//
// Rank 0 prints one JSON object per (mode, SNR point) with the Wilson 95 % interval of the FER, then one summary line with the
// per-rank run times (scaling efficiency = mean / max of the ranks' times: ranks never wait for each other before the final sum).
#include <dlfcn.h>
#include <unistd.h>

#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "pu/pu_capi.h"

namespace {

struct NcclId { char internal[128]; };
struct Nccl {
    int (*GetUniqueId)(NcclId*) = nullptr;
    int (*CommInitRank)(void**, int, NcclId, int) = nullptr;
    int (*CommDestroy)(void*) = nullptr;
    bool load() {
        void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (!h) return false;
        GetUniqueId = reinterpret_cast<int (*)(NcclId*)>(dlsym(h, "ncclGetUniqueId"));
        CommInitRank = reinterpret_cast<int (*)(void**, int, NcclId, int)>(dlsym(h, "ncclCommInitRank"));
        CommDestroy = reinterpret_cast<int (*)(void*)>(dlsym(h, "ncclCommDestroy"));
        return GetUniqueId && CommInitRank && CommDestroy;
    }
};

const char* kWaveform[] = {"OFDM", "OFDM_SC", "OFDM_CHIRP", "DPSK", "DPSK_ACQ", "MC_DPSK", "MC_DPSK_CHIRP"};
const char* kChannel[] = {"awgn", "good", "moderate", "poor", "flutter", "itu_good", "itu_moderate", "itu_poor", "itu_flutter"};
const char* kRate[] = {"R1/4", "R1/3", "R1/2", "R2/3", "R3/4", "R5/6", "R7/8"};
const char* mod_name(unsigned m) {
    switch (m) {
        case PU_MOD_DBPSK: return "DBPSK"; case PU_MOD_BPSK: return "BPSK"; case PU_MOD_DQPSK: return "DQPSK"; case PU_MOD_QPSK: return "QPSK";
        case PU_MOD_D8PSK: return "D8PSK"; case PU_MOD_QAM16: return "16QAM"; case PU_MOD_QAM32: return "32QAM"; case PU_MOD_QAM64: return "64QAM";
        case PU_MOD_QAM256: return "256QAM"; default: return "?";
    }
}
unsigned payload_of(unsigned rate) {   // floor(k / 8): k = 162, 216, 324, 432, 486, 540 (LDPCDecoder::getCodeParams, ldpc_decoder.cpp:21-36)
    static const unsigned k[] = {162, 216, 324, 432, 486, 540, 567};
    return k[rate] / 8;
}

// Acquired frames are surrounded by silence as the reference's tools do (test_iwaveform.cpp:396-459: 1.5 s before, 1 s behind; here 10 ms
// and 50 ms -- enough for the channel's path delays and the acquisition's jitter, without tripling the search buffers): without a tail
// the delayed path pushes the last symbol out of the buffer and the receiver hands out fewer than 648 soft bits.
constexpr unsigned kLead = 480, kTail = 2400;

pu_sweep_mode ofdm_mode(unsigned wf, unsigned fft, unsigned mod, unsigned rate, unsigned ch, float s0, float ds, unsigned n, bool fast) {
    pu_sweep_mode m{};
    const bool diff = mod == PU_MOD_DBPSK || mod == PU_MOD_DQPSK || mod == PU_MOD_D8PSK;
    m.waveform = wf;
    // ModemConfig defaults (include/ultra/types.hpp:139-195) for 512, presets::nvis_mode() (:342-355) for 1024; coherent modes carry
    // pilots (tools/test_mode_snr.cpp:30, tools/test_nvis_mode.cpp:209-212)
    m.ofdm = fft == 512 ? pu_modem_config{48000, 1500, 512, 30, 1, 4, 2, diff ? 0u : 1u, mod, rate, 40.0f, 0.0f}
                        : pu_modem_config{48000, 1500, 1024, 59, 1, 0, diff ? 2u : 4u, diff ? 0u : 1u, mod, rate, 40.0f, 0.0f};
    m.code_rate = rate; m.payload_bytes = payload_of(rate); m.channel = ch; m.n_snr = n; m.snr_first_db = s0; m.snr_step_db = ds;
    m.peak = wf == PU_WF_OFDM ? 0.0f : 0.5f;
    m.precision = fast ? PU_PRECISION_FAST : PU_PRECISION_EXACT;
    if (wf != PU_WF_OFDM) { m.lead_samples = kLead; m.tail_samples = kTail; }
    return m;
}
pu_sweep_mode dpsk_mode(unsigned wf, unsigned mod, unsigned rate, unsigned ch, float s0, float ds, unsigned n) {
    pu_sweep_mode m{};
    m.waveform = wf;
    m.dpsk = pu_dpsk_config{48000.0f, 1500.0f, 384, mod};            // 125 baud (tools/test_dpsk_snr.cpp:22)
    m.code_rate = rate; m.payload_bytes = payload_of(rate); m.channel = ch; m.n_snr = n; m.snr_first_db = s0; m.snr_step_db = ds; m.peak = 0.5f;
    if (wf == PU_WF_DPSK_ACQ) { m.lead_samples = kLead; m.tail_samples = kTail; }
    return m;
}
pu_sweep_mode mcdpsk_mode(unsigned wf, unsigned carriers, unsigned rate, unsigned ch, float s0, float ds, unsigned n) {
    pu_sweep_mode m{};
    m.waveform = wf;
    m.mcdpsk = pu_mcdpsk_config{48000.0f, 500.0f, 2500.0f, carriers, 512, 2, 8};   // MultiCarrierDPSKConfig defaults (multi_carrier_dpsk.hpp:26-60)
    m.code_rate = rate; m.payload_bytes = payload_of(rate); m.channel = ch; m.n_snr = n; m.snr_first_db = s0; m.snr_step_db = ds; m.peak = 0.5f;
    if (wf == PU_WF_MCDPSK_CHIRP) { m.lead_samples = kLead; m.tail_samples = kTail; }
    return m;
}

std::vector<pu_sweep_mode> make_table(const std::string& name, bool fast, unsigned frame_bytes) {
    std::vector<pu_sweep_mode> t;
    if (name == "frames") {
        // link-level FER: does a DATA frame of this many payload bytes arrive intact (several codewords in one OFDM frame)?
        std::vector<unsigned> sizes = frame_bytes ? std::vector<unsigned>{frame_bytes} : std::vector<unsigned>{200, 1000};
        for (unsigned bytes : sizes)
            for (unsigned ch : {PU_CH_AWGN, PU_CH_GOOD, PU_CH_POOR}) {
                const float step = ch == PU_CH_AWGN ? 1.0f : 2.0f;
                pu_sweep_mode rows[] = {ofdm_mode(PU_WF_OFDM, 512, PU_MOD_DQPSK, PU_RATE_1_2, ch, -2, step, 12, fast),
                                        ofdm_mode(PU_WF_OFDM, 512, PU_MOD_QAM16, PU_RATE_1_2, ch, 6, step, 12, fast),
                                        ofdm_mode(PU_WF_OFDM, 1024, PU_MOD_QAM32, PU_RATE_3_4, ch, 10, step, 12, fast),
                                        ofdm_mode(PU_WF_OFDM_CHIRP, 512, PU_MOD_DQPSK, PU_RATE_1_2, ch, 0, step, 12, fast)};
                for (pu_sweep_mode& m : rows) {
                    m.frame_payload_bytes = bytes;
                    t.push_back(m);
                }
            }
    } else if (name == "smoke") {
        t.push_back(ofdm_mode(PU_WF_OFDM, 512, PU_MOD_DQPSK, PU_RATE_1_2, PU_CH_AWGN, -4, 1, 13, fast));
        t.push_back(ofdm_mode(PU_WF_OFDM, 1024, PU_MOD_QAM32, PU_RATE_3_4, PU_CH_GOOD, 8, 2, 6, fast));
        t.push_back(dpsk_mode(PU_WF_DPSK, 1, PU_RATE_1_4, PU_CH_POOR, -11, 4, 8));
        t.push_back(mcdpsk_mode(PU_WF_MCDPSK, 8, PU_RATE_1_2, PU_CH_MODERATE, -2, 2, 8));
    } else if (name == "reduced") {
        // one mode per waveform family, the four channel conditions of the regression matrix, genie-timed and acquired variants
        for (unsigned ch : {PU_CH_AWGN, PU_CH_GOOD, PU_CH_MODERATE, PU_CH_POOR}) {
            t.push_back(ofdm_mode(PU_WF_OFDM, 512, PU_MOD_DQPSK, PU_RATE_1_2, ch, -4, 1, 16, fast));
            t.push_back(ofdm_mode(PU_WF_OFDM, 512, PU_MOD_QAM16, PU_RATE_1_2, ch, 4, 1, 16, fast));
            t.push_back(ofdm_mode(PU_WF_OFDM, 1024, PU_MOD_QAM32, PU_RATE_3_4, ch, 8, 1, 16, fast));
            t.push_back(mcdpsk_mode(PU_WF_MCDPSK, 8, PU_RATE_1_2, ch, -6, 1, 16));
            t.push_back(dpsk_mode(PU_WF_DPSK, 1, PU_RATE_1_4, ch, -11, 2, 15));
        }
        t.push_back(ofdm_mode(PU_WF_OFDM_SC, 512, PU_MOD_DQPSK, PU_RATE_1_2, PU_CH_AWGN, 10, 3, 8, fast));   // Schmidl-Cox needs its 0.8 plateau
        // the chirp-acquired rows of tests/regression_matrix.sh:139-243 with their tuning error (--cfo 0 / 30 / 50 / -30): the tools'
        // FFT-Hilbert injector on the clean TX audio (pu_sweep_mode.cfo_hz)
        for (float cfo : {0.0f, 30.0f, 50.0f}) {
            pu_sweep_mode m = ofdm_mode(PU_WF_OFDM_CHIRP, 512, PU_MOD_DQPSK, PU_RATE_1_2, PU_CH_AWGN, 5, 1, 16, fast);   // "--snr 17 --cfo 30/50 awgn ofdm_chirp"
            m.cfo_hz = cfo;
            t.push_back(m);
        }
        for (unsigned ch : {PU_CH_AWGN, PU_CH_MODERATE, PU_CH_POOR})
            for (float cfo : {0.0f, 30.0f, -30.0f}) {
                pu_sweep_mode m = mcdpsk_mode(PU_WF_MCDPSK_CHIRP, 8, PU_RATE_1_2, ch, -6, 1, 22);                       // "--snr 5/0/10/15 --cfo 30 mc_dpsk"
                m.cfo_hz = cfo;
                t.push_back(m);
            }
        {
            pu_sweep_mode m = ofdm_mode(PU_WF_OFDM_CHIRP, 512, PU_MOD_DQPSK, PU_RATE_1_4, PU_CH_MODERATE, 5, 1, 16, fast);   // "--snr 15 --cfo 30 moderate --rate r1_4"
            m.cfo_hz = 30.0f;
            t.push_back(m);
        }
    } else {   // config5: all waveforms x 5 rates x 40 SNR points in 1 dB steps, the grid shifted per family (-8, -14, -28 dB upwards)
        const unsigned rates[] = {PU_RATE_1_4, PU_RATE_1_2, PU_RATE_2_3, PU_RATE_3_4, PU_RATE_5_6};
        for (unsigned r : rates) {
            for (unsigned mod : {PU_MOD_DBPSK, PU_MOD_DQPSK, PU_MOD_D8PSK, PU_MOD_BPSK, PU_MOD_QPSK, PU_MOD_QAM16, PU_MOD_QAM32, PU_MOD_QAM64})
                t.push_back(ofdm_mode(PU_WF_OFDM, 512, mod, r, PU_CH_GOOD, -8, 1, 40, fast));
            for (unsigned mod : {PU_MOD_DQPSK, PU_MOD_QAM16, PU_MOD_QAM32, PU_MOD_QAM64})
                t.push_back(ofdm_mode(PU_WF_OFDM, 1024, mod, r, PU_CH_GOOD, -8, 1, 40, fast));
            t.push_back(ofdm_mode(PU_WF_OFDM_CHIRP, 512, PU_MOD_DQPSK, r, PU_CH_GOOD, -8, 1, 40, fast));
            for (unsigned nc : {3u, 5u, 8u, 13u, 20u}) t.push_back(mcdpsk_mode(PU_WF_MCDPSK_CHIRP, nc, r, PU_CH_POOR, -14, 1, 40));
            for (unsigned mod : {0u, 1u, 2u}) t.push_back(dpsk_mode(PU_WF_DPSK_ACQ, mod, r, PU_CH_POOR, -28, 1, 40));
        }
    }
    return t;
}

const char* arg(int argc, char** argv, const char* name, const char* dflt) {
    for (int i = 1; i + 1 < argc; ++i)
        if (!strcmp(argv[i], name)) return argv[i + 1];
    return dflt;
}
bool flag(int argc, char** argv, const char* name) {
    for (int i = 1; i < argc; ++i)
        if (!strcmp(argv[i], name)) return true;
    return false;
}
int env_int(const char* n, int d) { const char* v = getenv(n); return v ? atoi(v) : d; }

}  // namespace

int main(int argc, char** argv) {
    const int rank = env_int("RANK", 0), world = env_int("WORLD_SIZE", 1), local = env_int("LOCAL_RANK", rank);
    const std::string table = arg(argc, argv, "--table", "smoke");
    const bool fresh = flag(argc, argv, "--fresh");      // a new payload per trial in every mode (TX, chirp pair and tuning error on the GPU inside the batch)
    const std::string manifest = arg(argc, argv, "--manifest", "");
    const std::string out_path = arg(argc, argv, "--out", "");
    const std::string rdv = arg(argc, argv, "--rendezvous", manifest.empty() ? "/tmp" : manifest.c_str());
    const bool fast = strcmp(arg(argc, argv, "--precision", "fast"), "exact") != 0;
    // equal on all ranks of one launch, different between launches: the launcher's pid (torchrun's agent is every worker's parent)
    const unsigned long long run_id = strtoull(arg(argc, argv, "--run-id", "0"), nullptr, 0)
                                          ? strtoull(arg(argc, argv, "--run-id", "0"), nullptr, 0)
                                          : (static_cast<unsigned long long>(getppid()) << 16) ^ static_cast<unsigned long long>(env_int("MASTER_PORT", 0));

    pu_ctx* ctx = nullptr;
    if (pu_init(local, &ctx) != PU_OK) { fprintf(stderr, "pu_sweep[%d]: %s\n", rank, pu_last_error()); return 2; }

    // ---- NCCL communicator (only for the final sum): rank 0 publishes the unique id through a file
    void* comm = nullptr;
    Nccl nccl;
    if (world > 1) {
        if (!nccl.load()) { fprintf(stderr, "pu_sweep[%d]: libnccl.so.2 not found\n", rank); return 2; }
        NcclId id{};
        char path[512];
        snprintf(path, sizeof path, "%s/pu_sweep-nccl-%llx.id", rdv.c_str(), run_id);
        if (rank == 0) {
            if (nccl.GetUniqueId(&id) != 0) { fprintf(stderr, "pu_sweep: ncclGetUniqueId failed\n"); return 2; }
            const std::string tmp = std::string(path) + ".tmp";
            FILE* f = fopen(tmp.c_str(), "wb");
            if (!f || fwrite(&id, sizeof id, 1, f) != 1) { fprintf(stderr, "pu_sweep: cannot write %s\n", tmp.c_str()); return 2; }
            fclose(f);
            rename(tmp.c_str(), path);
        } else {
            for (int tries = 0;; ++tries) {
                FILE* f = fopen(path, "rb");
                if (f) {
                    const bool ok = fread(&id, sizeof id, 1, f) == 1;
                    fclose(f);
                    if (ok) break;
                }
                if (tries > 3000) { fprintf(stderr, "pu_sweep[%d]: timed out waiting for %s\n", rank, path); return 2; }
                std::this_thread::sleep_for(std::chrono::milliseconds(20));
            }
        }
        if (nccl.CommInitRank(&comm, world, id, rank) != 0) { fprintf(stderr, "pu_sweep[%d]: ncclCommInitRank failed\n", rank); return 2; }
        if (rank == 0) remove(path);
    }

    const unsigned frame_bytes = static_cast<unsigned>(atoi(arg(argc, argv, "--frame-bytes", "0")));
    std::vector<pu_sweep_mode> modes = make_table(table, fast, frame_bytes);
    if (fresh)
        for (auto& m : modes) m.fresh_payloads = 1;
    if (flag(argc, argv, "--interleave"))
        for (auto& m : modes) {
            if (m.waveform <= PU_WF_OFDM_CHIRP) {
                pu_ofdm* h = nullptr;
                if (pu_ofdm_create(ctx, &m.ofdm, &h) != PU_OK) { fprintf(stderr, "pu_sweep[%d]: %s\n", rank, pu_last_error()); return 2; }
                m.interleave_bps = static_cast<uint32_t>(pu_ofdm_bits_per_symbol(h));
                pu_ofdm_destroy(h);
            } else if (m.waveform >= PU_WF_MCDPSK) {
                m.interleave_bps = m.mcdpsk.num_carriers * m.mcdpsk.bits_per_symbol;
            }
        }
    pu_sweep_desc d{};
    d.modes = modes.data();
    d.n_modes = static_cast<uint32_t>(modes.size());
    d.pool = static_cast<uint32_t>(atoi(arg(argc, argv, "--pool", "32")));
    d.trials_per_point = strtoull(arg(argc, argv, "--trials", "4096"), nullptr, 0);
    d.block_trials = static_cast<uint32_t>(atoi(arg(argc, argv, "--block", "2048")));
    d.rank = static_cast<uint32_t>(rank);
    d.world = static_cast<uint32_t>(world);
    d.manifest_dir = manifest.empty() ? nullptr : manifest.c_str();
    d.max_units = strtoull(arg(argc, argv, "--max-units", "0"), nullptr, 0);
    d.run_id = run_id;
    const uint32_t n_points = pu_sweep_point_count(&d);
    if (n_points == 0) { fprintf(stderr, "pu_sweep: invalid table\n"); return 2; }

    // --raw: pre-decoder counters {soft_bits, erasures, bit_errors, strong_errors} per point (pu_linksim_run_raw), summed with the rest
    const bool want_raw = flag(argc, argv, "--raw");
    std::vector<uint64_t> counters(static_cast<size_t>(n_points) * 6 + 3 * world + (want_raw ? static_cast<size_t>(n_points) * 4 : 0), 0);
    uint64_t* raw = want_raw ? counters.data() + static_cast<size_t>(n_points) * 6 + 3 * world : nullptr;
    pu_sweep_stats st{};
    const pu_status rs = pu_linksim_run_raw(ctx, &d, counters.data(), raw, &st);
    if (rs != PU_OK) { fprintf(stderr, "pu_sweep[%d]: pu_linksim_run: %s: %s\n", rank, pu_status_string(rs), pu_last_error()); return 3; }
    // per-rank run time / frames / launches ride behind the counters: slot `rank` is this rank's, the sum fills in the others
    uint64_t* tail = counters.data() + static_cast<size_t>(n_points) * 6;
    tail[rank] = static_cast<uint64_t>(st.seconds * 1e6);
    tail[world + rank] = st.frames_run;
    tail[2 * world + rank] = pu_kernel_launches(ctx);
    if (pu_counters_allreduce(ctx, counters.data(), counters.size(), comm, PU_MEM_HOST, nullptr) != PU_OK) {
        fprintf(stderr, "pu_sweep[%d]: %s\n", rank, pu_last_error());
        return 3;
    }

    if (rank == 0) {
        FILE* out = out_path.empty() ? stdout : fopen(out_path.c_str(), "w");
        if (!out) out = stdout;
        uint32_t at = 0;
        uint64_t frames_all = 0;
        for (uint32_t m = 0; m < d.n_modes; ++m) {
            const pu_sweep_mode& md = modes[m];
            const bool is_ofdm = md.waveform <= PU_WF_OFDM_CHIRP, is_dpsk = md.waveform == PU_WF_DPSK || md.waveform == PU_WF_DPSK_ACQ;
            char desc[96];
            if (is_ofdm) snprintf(desc, sizeof desc, "%u-FFT %s%s", md.ofdm.fft_size, mod_name(md.ofdm.modulation), md.ofdm.use_pilots ? " pilots" : "");
            else if (is_dpsk) snprintf(desc, sizeof desc, "%s 125 baud", md.dpsk.modulation == 0 ? "DBPSK" : md.dpsk.modulation == 1 ? "DQPSK" : "D8PSK");
            else snprintf(desc, sizeof desc, "%u carriers DQPSK", md.mcdpsk.num_carriers);
            char il[40] = "";
            if (md.interleave_bps) snprintf(il, sizeof il, ", \"interleave_bps\": %u", md.interleave_bps);
            for (uint32_t s = 0; s < md.n_snr; ++s, ++at) {
                const uint64_t* c = &counters[static_cast<size_t>(at) * 6];
                char rw[192] = "";
                if (raw) {      // raw BER over the soft bits that are not erasures; strong errors: |llr| >= 10 (the demappers' clip)
                    const uint64_t* r = raw + static_cast<size_t>(at) * 4;
                    snprintf(rw, sizeof rw, ", \"soft_bits\": %llu, \"raw_bit_errors\": %llu, \"raw_ber\": %.6g, \"erasure_rate\": %.6g, \"strong_error_share\": %.6g",
                             (unsigned long long)r[0], (unsigned long long)r[2], r[0] > r[1] ? double(r[2]) / double(r[0] - r[1]) : 0.0,
                             r[0] ? double(r[1]) / r[0] : 0.0, r[2] ? double(r[3]) / r[2] : 0.0);
                }
                double lo, hi;
                pu_wilson_interval(c[1], c[0], 1.96, &lo, &hi);
                frames_all += c[0];
                if (md.frame_payload_bytes) {     // whole-frame counters {frames, frame_errors, codewords_failed, codewords, header_failures, 0}
                    fprintf(out, "{\"mode\": %u, \"waveform\": \"%s\", \"modem\": \"%s\", \"code_rate\": \"%s\", \"channel\": \"%s\", \"cfo_hz\": %.1f, \"snr_db\": %.2f, "
                                 "\"frame_payload_bytes\": %u, \"codewords\": %llu, \"frames\": %llu, \"frame_errors\": %llu, \"fer\": %.6g, \"fer_ci95\": [%.6g, %.6g], "
                                 "\"codeword_fail_rate\": %.6g, \"header_fail_rate\": %.6g%s%s}\n",
                            m, kWaveform[md.waveform], desc, kRate[md.code_rate], kChannel[md.channel], md.cfo_hz, md.snr_first_db + s * md.snr_step_db,
                            md.frame_payload_bytes, (unsigned long long)(c[0] ? c[3] / c[0] : 0), (unsigned long long)c[0], (unsigned long long)c[1],
                            c[0] ? double(c[1]) / c[0] : 0.0, lo, hi, c[3] ? double(c[2]) / c[3] : 0.0, c[0] ? double(c[4]) / c[0] : 0.0, il, rw);
                    continue;
                }
                fprintf(out, "{\"mode\": %u, \"waveform\": \"%s\", \"modem\": \"%s\", \"code_rate\": \"%s\", \"channel\": \"%s\", \"cfo_hz\": %.1f, \"snr_db\": %.2f, "
                             "\"frames\": %llu, \"frame_errors\": %llu, \"fer\": %.6g, \"fer_ci95\": [%.6g, %.6g], \"ber\": %.6g, \"decode_fail\": %.6g, "
                             "\"avg_iters\": %.4g%s%s}\n",
                        m, kWaveform[md.waveform], desc, kRate[md.code_rate], kChannel[md.channel], md.cfo_hz, md.snr_first_db + s * md.snr_step_db,
                        (unsigned long long)c[0], (unsigned long long)c[1], c[0] ? double(c[1]) / c[0] : 0.0, lo, hi, c[3] ? double(c[2]) / c[3] : 0.0,
                        c[0] ? double(c[4]) / c[0] : 0.0, c[0] ? double(c[5]) / c[0] : 0.0, il, rw);
            }
        }
        double tmax = 0, tsum = 0;
        uint64_t frames_run = 0, launches = 0;
        std::string per_rank = "[";
        for (int r = 0; r < world; ++r) {
            const double t = tail[r] * 1e-6;
            tmax = t > tmax ? t : tmax;
            tsum += t;
            frames_run += tail[world + r];
            launches += tail[2 * world + r];
            char b[32];
            snprintf(b, sizeof b, "%s%.3f", r ? ", " : "", t);
            per_rank += b;
        }
        per_rank += "]";
        fprintf(out, "{\"summary\": true, \"table\": \"%s\", \"modes\": %u, \"points\": %u, \"trials_per_point\": %llu, \"world\": %d, "
                     "\"units\": %llu, \"units_resumed\": %llu, \"frames_counted\": %llu, \"frames_run\": %llu, \"seconds_per_rank\": %s, "
                     "\"seconds\": %.3f, \"frames_per_s\": %.6g, \"balance_efficiency\": %.4f, \"gpu_launches\": %llu, \"precision\": \"%s\", \"fresh_payloads\": %s, "
                     "\"rank0_seconds\": {\"setup\": %.3f, \"wait\": %.3f, \"fill\": %.3f, \"enqueue\": %.3f}}\n",
                table.c_str(), d.n_modes, n_points, (unsigned long long)d.trials_per_point, world, (unsigned long long)st.units_total,
                (unsigned long long)st.units_resumed, (unsigned long long)frames_all, (unsigned long long)frames_run, per_rank.c_str(), tmax,
                tmax > 0 ? frames_run / tmax : 0.0, tmax > 0 ? tsum / world / tmax : 1.0, (unsigned long long)launches, fast ? "fast" : "exact", fresh ? "true" : "false",
                st.setup_seconds, st.wait_seconds, st.fill_seconds, st.enqueue_seconds);
        if (out != stdout) fclose(out);
    }
    if (comm) nccl.CommDestroy(comm);
    pu_destroy(ctx);
    return 0;
}
