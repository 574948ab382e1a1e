/* include/pu/pu_capi.h — C ABI of libpu_b200.so, the B200-native receive-chain hot path of ProjectUltra.
 *
 * This is the drop-in boundary (SURVEY §8b): plain pointers and sizes, no C++ or torch types.  Every entry
 * point cites the reference interface it replaces (paths relative to the reference tree).  The C++20 classes
 * in include/pu/pu_dropin.hpp wrap these calls to present the reference's own class surface
 * (ultra::LDPCDecoder, ultra::OFDMDemodulator, ultra::ChannelInterleaver, ultra::IWaveform) unchanged;
 * INTEGRATION.md shows the binding a reference maintainer would add.
 *
 * Conventions
 *  - status codes, never exceptions (the reference decode path does not throw: SURVEY §8b "Errors");
 *  - outputs are caller-allocated; `space` says whether ALL data pointers of a call are host or device memory;
 *  - `stream` is a cudaStream_t passed as void*.  With PU_MEM_DEVICE the call only enqueues work on `stream`
 *    (NULL = the CUDA default stream, as in the runtime API); with PU_MEM_HOST it stages through pinned memory
 *    on `stream` (NULL = a stream owned by the context) and returns when the outputs are valid;
 *  - there is NO CPU fallback: every compute entry point fails with PU_ERR_CUDA when no sm_100 device is usable.
 */
#ifndef PU_CAPI_H
#define PU_CAPI_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define PU_API __declspec(dllexport)
#else
#define PU_API __attribute__((visibility("default")))
#endif

typedef enum {
    PU_OK = 0,
    PU_ERR_INVALID = 1,      /* bad argument */
    PU_ERR_CUDA = 2,         /* CUDA runtime / launch failure, or no usable device */
    PU_ERR_NOMEM = 3,
    PU_ERR_UNSUPPORTED = 4   /* configuration outside the implemented hot path */
} pu_status;

typedef enum { PU_MEM_HOST = 0, PU_MEM_DEVICE = 1 } pu_memspace;

/* ultra::Modulation, include/ultra/types.hpp:27-39 */
enum { PU_MOD_DBPSK = 0, PU_MOD_BPSK = 1, PU_MOD_DQPSK = 2, PU_MOD_QPSK = 3, PU_MOD_D8PSK = 4, PU_MOD_QAM8 = 5,
       PU_MOD_QAM16 = 6, PU_MOD_QAM32 = 7, PU_MOD_QAM64 = 8, PU_MOD_QAM256 = 10 };
/* ultra::CodeRate, include/ultra/types.hpp:92-101 */
enum { PU_RATE_1_4 = 0, PU_RATE_1_3 = 1, PU_RATE_1_2 = 2, PU_RATE_2_3 = 3, PU_RATE_3_4 = 4, PU_RATE_5_6 = 5,
       PU_RATE_7_8 = 6 };
#define PU_LDPC_N 648 /* protocol::v2::LDPC_CODEWORD_BITS, src/protocol/frame_v2.hpp:546 */

/* POD mirror of ultra::ModemConfig (include/ultra/types.hpp:139-234), the fields the receive path reads. */
typedef struct {
    uint32_t sample_rate;   /* 48000 */
    uint32_t center_freq;   /* 1500 */
    uint32_t fft_size;      /* 512 | 1024 */
    uint32_t num_carriers;  /* 30 | 59 */
    uint32_t cp_mode;       /* CyclicPrefixMode: 0 SHORT(32) 1 MEDIUM(48) 2 LONG(64), x fft_size/512 */
    uint32_t symbol_guard;
    uint32_t pilot_spacing;
    uint32_t use_pilots;
    uint32_t modulation;    /* PU_MOD_* */
    uint32_t code_rate;     /* PU_RATE_* */
    float output_scale;     /* TX only (40.0) */
    float tx_cfo_hz;        /* TX only */
} pu_modem_config;

typedef struct pu_ctx pu_ctx;
typedef struct pu_ldpc pu_ldpc;
typedef struct pu_ofdm pu_ofdm;

/* ---------------------------------------------------------------- context */
PU_API int pu_abi_version(void);
PU_API const char* pu_status_string(pu_status s);
PU_API const char* pu_last_error(void);                 /* thread-local detail of the last failing call */
PU_API pu_status pu_init(int device, pu_ctx** out);    /* one context per GPU / per process rank */
PU_API void pu_destroy(pu_ctx* ctx);
PU_API int pu_device_sm_count(const pu_ctx* ctx);
PU_API pu_status pu_synchronize(pu_ctx* ctx, void* stream);
PU_API uint64_t pu_kernel_launches(const pu_ctx* ctx);  /* kernels launched through this context so far */
/* bytes copied host->device / device->host by pu_receive_decode_batch(PU_MEM_HOST) through this context so far */
PU_API void pu_transfer_bytes(const pu_ctx* ctx, uint64_t* h2d_bytes, uint64_t* d2h_bytes);

/* ---------------------------------------------------------------- LDPC decoder
 * Replaces ultra::LDPCDecoder (include/ultra/fec.hpp:48-77; src/fec/ldpc_decoder.cpp). */
/* LDPCDecoder::LDPCDecoder(CodeRate) + setMaxIterations, ldpc_decoder.cpp:262-263,448-450 (default 50, :43) */
PU_API pu_status pu_ldpc_create(pu_ctx* ctx, int code_rate, int max_iter, pu_ldpc** out);
PU_API void pu_ldpc_destroy(pu_ldpc* h);
PU_API pu_status pu_ldpc_set_rate(pu_ldpc* h, int code_rate);      /* LDPCDecoder::setRate, :438-442 */
PU_API pu_status pu_ldpc_set_max_iterations(pu_ldpc* h, int n);    /* LDPCDecoder::setMaxIterations, :448-450 */
PU_API int pu_ldpc_rate(const pu_ldpc* h);                         /* LDPCDecoder::getRate, :444-446 */
PU_API int pu_ldpc_info_bits(const pu_ldpc* h);                    /* k of getCodeParams, :21-36 */
PU_API int pu_ldpc_num_edges(const pu_ldpc* h);                    /* edges of H incl. identity (SURVEY App. C) */
/* H row i as variable indices in stored order (for inspection/tests); returns the degree or -1 */
PU_API int pu_ldpc_row(const pu_ldpc* h, int check, int32_t* vars, int cap);
/* B independent codewords of 648 LLRs (+ => bit 0).  One decodeBP each (ldpc_decoder.cpp:153-259):
 * info_bytes[b*info_stride ...] = k info bits MSB-first, last byte left-justified; ok[b] = lastDecodeSuccess();
 * iters[b] = lastIterations() (0-based converging iteration, max_iter on failure).  ok / iters may be NULL.
 * llr_stride is in floats (>= 648). */
PU_API pu_status pu_ldpc_decode_batch(pu_ldpc* h, const float* llr, size_t llr_stride, size_t B,
                                      uint8_t* info_bytes, size_t info_stride, uint8_t* ok, int32_t* iters,
                                      pu_memspace space, void* stream);
/* LDPCDecoder::decodeSoft (ldpc_decoder.cpp:283-428) on HOST memory, including its multi-block rules:
 * <=648 LLRs -> one zero-padded block; otherwise full blocks concatenated at bit level and a zero-padded
 * trailing partial block.  *out_len receives the byte count; returns PU_ERR_INVALID if out_cap is too small. */
PU_API pu_status pu_ldpc_decode_soft(pu_ldpc* h, const float* llr, size_t n_llr, uint8_t* out, size_t out_cap,
                                     size_t* out_len, int* last_success, int* last_iters);
/* LDPCDecoder::decode (hard bits -> +-6 LLR, ldpc_decoder.cpp:267-281) on HOST memory */
PU_API pu_status pu_ldpc_decode_hard(pu_ldpc* h, const uint8_t* coded, size_t n_bytes, uint8_t* out, size_t out_cap,
                                     size_t* out_len, int* last_success, int* last_iters);
/* LDPCEncoder::encode (src/fec/ldpc_encoder.cpp:193-257), host side: TX stimulus for the link simulation */
PU_API pu_status pu_ldpc_encode(int code_rate, const uint8_t* data, size_t n_bytes, uint8_t* out, size_t out_cap,
                                size_t* out_len);

/* ---------------------------------------------------------------- interleavers (host tables)
 * ultra::ChannelInterleaver (include/ultra/fec.hpp:120-142; ldpc_decoder.cpp:547-620): perm[i] = (i*step)%total.
 * Writes perm[total]; interleave: out[perm[i]] = in[i]; deinterleave: out[inv[i]] = in[i]. */
PU_API pu_status pu_channel_interleaver_perm(size_t bits_per_symbol, size_t total_bits, uint32_t* perm,
                                             uint32_t* inverse_perm, size_t* step);
/* ultra::Interleaver (fec.hpp:85-107; ldpc_decoder.cpp:454-464): perm[i] = (i%cols)*rows + i/cols */
PU_API pu_status pu_block_interleaver_perm(size_t rows, size_t cols, uint32_t* perm);
/* ChannelInterleaver(bits_per_symbol, 648)::deinterleave on the soft bits of any receiver, the step RxPipeline takes between getSoftBits
 * and decodeSoft, 648 soft bits at a time: IN PLACE on llr[b*llr_stride + c*648 .. + 648) for b < B and c < n_blocks, every block on
 * its own (out[k] = in[k * step mod 648]).  n_blocks * 648 <= llr_stride; the columns beyond n_blocks * 648 are not written.  A block
 * of zeros (an erasure) stays zeros.  PU_MEM_HOST stages the first n_blocks * 648 soft bits of every row (csrc/interleave.cu). */
PU_API pu_status pu_llr_deinterleave_batch(pu_ctx* ctx, float* llr, size_t B, size_t llr_stride, size_t n_blocks,
                                           size_t bits_per_symbol, pu_memspace space, void* stream);

/* ---------------------------------------------------------------- OFDM demodulator (presynced path)
 * Replaces ultra::OFDMDemodulator (include/ultra/ofdm.hpp:58-127) on the externally-timed path that
 * OFDMChirpWaveform::process drives (src/waveform/ofdm_chirp_waveform.cpp:185-199):
 *     reset(); setFrequencyOffset[WithPhase](cfo, phase); processPresynced(span, training); getSoftBits()...  */
/* OFDMDemodulator::OFDMDemodulator(const ModemConfig&), src/ofdm/demodulator.cpp:26-43,457-458.
 * PU_ERR_UNSUPPORTED for fft sizes other than 512/1024, QAM8/AUTO, or adaptive LMS/RLS equalisation
 * (ModemConfig::adaptive_eq_enabled, default off, is not part of pu_modem_config). */
PU_API pu_status pu_ofdm_create(pu_ctx* ctx, const pu_modem_config* cfg, pu_ofdm** out);
PU_API void pu_ofdm_destroy(pu_ofdm* h);
PU_API int pu_ofdm_symbol_samples(const pu_ofdm* h);   /* ModemConfig::getSymbolDuration, types.hpp:211-213 */
PU_API int pu_ofdm_data_carriers(const pu_ofdm* h);
PU_API int pu_ofdm_pilot_carriers(const pu_ofdm* h);
PU_API int pu_ofdm_bits_per_symbol(const pu_ofdm* h);  /* OFDMModulator::bitsPerSymbol, modulator.cpp:342-346 */
/* Diagnostic (no reference counterpart): which kernel the last pu_ofdm_presynced_batch / pu_receive_decode_batch launch on
 * this handle used: 0 = none yet, 1 = general presynced kernel (ofdm_demod.cu), 2 = warp-FFT kernel for differential
 * no-pilot modes (ofdm_diff.cu), 3 = persistent TMA-staged packed-fp32 512-FFT kernel (ofdm_diff512.cu), 4 = general presynced
 * kernel in its one-frame-per-warp form (ofdm_demod.cu, WARPG), 5 = FMA-contracted form of kernel 3 (ofdm_fast512.cu,
 * PU_PRECISION_FAST), 6 = kernel 4 with FMA butterflies and MUFU sin/cos in the CFO rotator (PU_PRECISION_FAST). */
PU_API int pu_ofdm_last_kernel(const pu_ofdm* h);
/* Arithmetic contract of the receive kernels of this handle (no reference counterpart; the reference has one build).
 *   PU_PRECISION_EXACT (default): FFT bins, channel estimate, equalised symbols bit-identical to the reference's unfused
 *     radix-2 fp32 arithmetic (src/dsp/fft.cpp:89-121, compiled without FMA contraction), LLR words >= 99.99 % identical.
 *   PU_PRECISION_FAST: BASELINE.json's own bar -- LLRs within 1e-4 relative (of max(|LLR|, 0.5)), saturated LLRs exactly
 *     +-10, decoded bytes identical on every frame the reference decodes with margin; butterflies are fused multiply-adds.
 *     The 512-FFT differential no-pilot modes at zero CFO take ofdm_fast512.cu; every other whole-frame call (pilots, coherent QAM,
 *     CFO, 1024-FFT pilot modes, acquired frames) takes the general warp kernel with FMA butterflies and MUFU sin/cos in the CFO
 *     rotator (the rotator's phases stay the reference's float recurrence); the remaining kernels (1024-FFT differential
 *     no-pilot, debug dumps) have no fast form and run exact. */
typedef enum pu_precision { PU_PRECISION_EXACT = 0, PU_PRECISION_FAST = 1 } pu_precision;
PU_API pu_status pu_ofdm_set_precision(pu_ofdm* h, pu_precision mode);
PU_API int pu_ofdm_get_precision(const pu_ofdm* h);
/* FFT bins of the used carriers, data carriers first then pilots (setupCarriers, demodulator.cpp:45-67) */
PU_API int pu_ofdm_carrier_bins(const pu_ofdm* h, int32_t* bins, int cap);
/* Fuse ChannelInterleaver(bits_per_symbol, total_bits)::deinterleave (ldpc_decoder.cpp:612-620) into the LLR
 * write address for the first total_bits LLRs of every frame; bits_per_symbol = 0 switches it off. */
PU_API pu_status pu_ofdm_set_deinterleave(pu_ofdm* h, size_t bits_per_symbol, size_t total_bits);
/* ChannelInterleaver(bits_per_symbol, 648)::interleave of every codeword in the transmitters of this handle: while it is set,
 * pu_ofdm_tx_batch and pu_frame_tx_batch interleave each 648-bit codeword on its own after LDPC encoding and before mapping, i.e.
 * transmitted bit j of a codeword is coded bit j * step^-1 mod 648 -- the waveform of pu_ofdm_tx on the interleaved bytes.
 * bits_per_symbol = 0 (the default) switches it off.  The receivers of the handle are unaffected: deinterleave with
 * pu_ofdm_set_deinterleave (first codeword, fused) or pu_llr_deinterleave_batch (any codeword), never both. */
PU_API pu_status pu_ofdm_set_tx_interleave(pu_ofdm* h, size_t bits_per_symbol);
/* B independent frames, each L samples starting at the first training symbol:
 *   samples [B][L]; cfo_hz[B] / cfo_phase[B] = arguments of setFrequencyOffsetWithPhase (demodulator.cpp:816-825),
 *   NULL meaning setFrequencyOffset(0) (:805-814);
 *   llr_out [B][llr_stride] receives the soft bits in getSoftBits() order (symbol-major, carrier, bit), truncated
 *   to llr_stride (648 = the first codeword, as tools/test_ofdm_chirp_pilots.cpp:244-246 consumes them);
 *   snr_db[B] = getEstimatedSNR(), final_cfo_hz[B] = getFrequencyOffset() after the frame (either may be NULL).
 * Each frame is demodulated by a fresh demodulator state, like one OFDMDemodulator object per frame. */
PU_API pu_status pu_ofdm_presynced_batch(pu_ofdm* h, const float* samples, size_t B, size_t L, int training_symbols,
                                         const float* cfo_hz, const float* cfo_phase, float* llr_out,
                                         size_t llr_stride, float* snr_db, float* final_cfo_hz,
                                         pu_memspace space, void* stream);
/* OFDMDemodulator::Impl::estimateCFOFromTraining(samples, training_symbols, 0) (src/ofdm/ofdm_sync.cpp:278-380) for B frames that start
 * at the first training symbol: the CFO processPresynced adopts when none was set (demodulator.cpp:918-925: after reset(), with
 * training_symbols >= 2).  cfo_hz[B]; 0 for training_symbols < 2, frames shorter than two symbols, or a correlation below 0.3.
 * A caller reproduces `reset(); processPresynced(span, n)` with this value as cfo_hz and phase 0 in pu_ofdm_presynced_batch. */
PU_API pu_status pu_ofdm_training_cfo_batch(pu_ofdm* h, const float* samples, size_t B, size_t L, int training_symbols,
                                            float* cfo_hz, pu_memspace space, void* stream);
/* ---------------------------------------------------------------- dual-chirp synchronisation (SURVEY 8f next-2)
 * sync::ChirpSync::detectDualChirp (src/sync/chirp_sync.hpp:349-506, configured as OFDMChirpWaveform::getChirpConfig,
 * src/waveform/ofdm_chirp_waveform.cpp:39-49) and the receive sequence of tools/test_iwaveform.cpp:127-160 on OFDM_CHIRP
 * frames: IWaveform::detectSync -> setFrequencyOffset(cfo) -> process(span from start_sample) -> getSoftBits, for B frames.
 *   sync_info[B][4]   = {detected, up_chirp_start, down_chirp_start, SyncResult::start_sample (training start) or -1}
 *   sync_values[B][4] = {cfo_hz, up correlation, down correlation, initial CFO-rotator phase}
 *   llr_out[B][llr_stride] (may be NULL: detection only), n_llr[B] = soft bits available (0 unless a codeword's worth, as
 *   OFDMChirpWaveform::process only collects them then); threshold <= 0 selects the callers' 0.15. */
PU_API pu_status pu_ofdm_chirp_receive_batch(pu_ofdm* h, const float* samples, size_t B, size_t L, float threshold,
                                             float* llr_out, size_t llr_stride, int32_t* n_llr, int32_t* sync_info,
                                             float* sync_values, float* snr_db, pu_memspace space, void* stream);
/* sync::ChirpSync::generate (chirp_sync.hpp:58-108), host side: [up chirp][gap][down chirp][gap]; out == NULL queries the length */
PU_API pu_status pu_chirp_generate(float sample_rate, float tx_cfo_hz, float* out, size_t out_cap, size_t* out_len);
/* Diagnostics of the two-tier chirp search (csrc/chirp_sync.cu) on the current device since the last call: templates searched, exact
 * verification rounds of the coarse search (one round = 16 coarse positions; a search that needs more than one had an unverified
 * position within the error bound of the best one) and exact runs of the fine search (16 consecutive positions each; 7 cover the
 * whole +-48 range).  Synchronises the device.  Any pointer may be NULL. */
PU_API pu_status pu_chirp_search_stats(uint64_t* searches, uint64_t* rounds, uint64_t* fine_runs);
/* sizeof of the public PODs, for bindings that mirror them by hand (ctypes, cgo, JNI): out[] = {pu_modem_config, pu_dpsk_config,
 * pu_mcdpsk_config, pu_channel_config, pu_sweep_mode, pu_sweep_desc, pu_sweep_stats, 0}.  Returns the number of entries filled. */
PU_API int pu_abi_sizes(uint32_t out[8]);

/* SM cycles the searches since the last call spent per phase (summed over frames, thread 0's clock): [0] low-pass + decimation,
 * [1] correlation estimates, [2] energies + ranking, [3] exact evaluation of the coarse leaders, [4] fine ranking, [5] exact fine runs. */
PU_API pu_status pu_chirp_phase_cycles(uint64_t cycles[8]);

/* ---------------------------------------------------------------- batched transmitter (SURVEY 8f next-3)
 * LDPCEncoder::encode (src/fec/ldpc_encoder.cpp:193-257, one 648-bit block, payload zero-padded to k bits) followed by
 * OFDMModulator::generateTrainingSymbols(2) (layout 0) or generatePreamble() (layout 1) + modulate()
 * (src/ofdm/modulator.cpp:348-580) for B payloads at once; peak > 0 rescales every frame to that peak amplitude as the
 * tools do (tools/test_mode_snr.cpp:52-56).  `code` supplies the code rate (its tables double as the encoder's).
 * out[B][out_stride] receives *frame_len samples per row; call with B = 0 to query *frame_len.  Waveforms are
 * bit-identical to pu_ldpc_encode + pu_ofdm_tx.  PU_MEM_HOST leaves each row's samples beyond *frame_len as they were. */
PU_API pu_status pu_ofdm_tx_batch(pu_ofdm* h, const pu_ldpc* code, const uint8_t* payload, size_t payload_stride,
                                  size_t payload_bytes, size_t B, int layout, float peak, float* out, size_t out_stride,
                                  size_t* frame_len, pu_memspace space, void* stream);
/* Multi-codeword frames (SURVEY 8f next-4): v2::encodeFrameWithLDPC (src/protocol/frame_v2.cpp:1079-1127: CW0 = the first
 * bytes_per_codeword frame bytes, CW1+ = {0xD5, index, next bytes_per_codeword - 2 bytes}, zero padded, each LDPC-encoded at the rate
 * of `code`) + OFDMModulator::generateTrainingSymbols(2) (layout 0) / generatePreamble() (layout 1) + modulate() over all
 * n_codewords x 648 coded bits back to back (src/ofdm/modulator.cpp:348-580: differential state carried across codewords, the last
 * symbol filled as far as the bits go), for B frames of frame_bytes bytes each (row b at frames + b * frame_stride).  peak > 0
 * rescales each frame as pu_ofdm_tx_batch does.  B = 0 queries *frame_len and *n_codewords (1..255; more is PU_ERR_INVALID).
 * Bit-identical to pu_frame_encode + pu_ofdm_tx(layout); pu_ofdm_tx_batch is its one-codeword case.  One CTA per frame, the coded
 * bits in shared memory (255 codewords: 20.7 KB). */
PU_API pu_status pu_frame_tx_batch(pu_ofdm* h, const pu_ldpc* code, const uint8_t* frames, size_t frame_stride, size_t frame_bytes,
                                   size_t B, int layout, float peak, float* out, size_t out_stride, size_t* frame_len,
                                   size_t* n_codewords, pu_memspace space, void* stream);

/* ---------------------------------------------------------------- OFDM acquisition (Schmidl-Cox path, SURVEY 8f next-1)
 * Replaces the SEARCHING state of ultra::OFDMDemodulator::process (src/ofdm/demodulator.cpp:474-600) with
 * Impl::hasMinimumEnergy / measureSchmidlCoxCorrelation / estimateCoarseCFO / refineLTSTiming
 * (src/ofdm/ofdm_sync.cpp:20-50,118-163,230-261,386-461) for B frames at once.  Row b of samples[B][L] is what a caller
 * would feed to process() in `chunk`-sample pieces (tools/test_mode_snr.cpp:65-70: 960); the search is replayed call
 * by call, so the result is the reference's for that chunking.  sync_info[B][4] = {synchronised (0/1),
 * getLastSyncOffset(), samples consumed up to the first data symbol, process() calls until sync};
 * coarse_cfo_hz[B] = the Schmidl-Cox CFO estimate.  sync_threshold <= 0 selects ModemConfig's default 0.80
 * (include/ultra/types.hpp:188).  PU_ERR_UNSUPPORTED for L > 40000 (the reference would trim its buffer). */
PU_API pu_status pu_ofdm_acquire_batch(pu_ofdm* h, const float* samples, size_t B, size_t L, size_t chunk,
                                       float sync_threshold, int32_t* sync_info, float* coarse_cfo_hz,
                                       pu_memspace space, void* stream);
/* ultra::OFDMDemodulator::process + getSoftBits (include/ultra/ofdm.hpp:58-127) on whole frames: acquisition as above,
 * then the SYNCED state (demodulator.cpp:665-690: per-symbol toBaseband / FFT / updateChannelEstimate / equalize /
 * demodulateSymbol with the coarse CFO, no LTS channel estimate) over every complete symbol after the preamble.
 * llr_out[B][llr_stride] (caller-zeroed rows; frames without sync stay untouched), n_llr[B] = soft bits available
 * (capped at llr_stride; < 648 is what the reference's tools count as a lost frame); sync_info / coarse_cfo_hz /
 * snr_db may be NULL.  The preamble search looks at the first 40 000 samples of a row (beyond them the reference trims its
 * buffer between calls); the data symbols behind a preamble found there run to the end of the row, whatever L is. */
PU_API pu_status pu_ofdm_process_batch(pu_ofdm* h, const float* samples, size_t B, size_t L, size_t chunk,
                                       float sync_threshold, float* llr_out, size_t llr_stride, int32_t* n_llr,
                                       int32_t* sync_info, float* coarse_cfo_hz, float* snr_db,
                                       pu_memspace space, void* stream);
/* One frame on HOST memory with per-symbol intermediates for stage-by-stage parity tests.  records holds, per
 * data symbol: bins[n_used] (re,im), channel_estimate[n_used] (re,im), equalized[n_data] (re,im),
 * carrier_noise_var[n_data], then 10 scalars {cfo used to mix, cfo after tracking, noise_variance,
 * timing_offset_samples, estimated_snr_linear, pilot_phase_correction re/im, carrier_phase_correction re/im,
 * snr_symbol_count}. */
PU_API pu_status pu_ofdm_presynced_debug(pu_ofdm* h, const float* samples, size_t L, int training_symbols,
                                         float cfo_hz, float cfo_phase, float* llr_out, size_t llr_cap,
                                         float* records, size_t records_cap, int* n_data_symbols);

/* ---------------------------------------------------------------- OFDM transmitter (host; TX stimulus)
 * OFDMModulator (include/ultra/ofdm.hpp:24-52; src/ofdm/modulator.cpp).  layout 0 = generateTrainingSymbols(2)
 * + modulate(data, cfg->modulation) -- the presynced frame of tools/test_ofdm_chirp_pilots.cpp:183-191;
 * layout 1 = generatePreamble() + modulate -- the Schmidl-Cox frame of tools/test_mode_snr.cpp:47-52.
 * Writes *out_len samples (also when out is too small, so callers can size the buffer). */
PU_API pu_status pu_ofdm_tx(const pu_modem_config* cfg, int layout, const uint8_t* data, size_t n_bytes,
                            float* out, size_t out_cap, size_t* out_len);

/* ---------------------------------------------------------------- single-carrier DPSK (externally timed)
 * Replaces ultra::DPSKDemodulator (src/psk/dpsk.hpp:309-1059) on frames whose data start is known (genie timing, or
 * the offset DPSKDemodulator::findPreamble returned -- Barker acquisition itself is SURVEY 8f next-2).
 * POD mirror of ultra::DPSKConfig (dpsk.hpp:42-50); modulation follows enum DPSKModulation (:31-35):
 * 0 DBPSK, 1 DQPSK, 2 D8PSK.  Pulse shaping (TX only) is on, as in the reference's default. */
typedef struct {
    float sample_rate;            /* 48000 */
    float carrier_freq;           /* 1500 */
    uint32_t samples_per_symbol;  /* 384 = 125 baud (tools/test_dpsk_snr.cpp:22), default 1536 */
    uint32_t modulation;
} pu_dpsk_config;
typedef struct pu_dpsk pu_dpsk;
PU_API pu_status pu_dpsk_create(pu_ctx* ctx, const pu_dpsk_config* cfg, pu_dpsk** out);   /* DPSKDemodulator ctor, :311-323 */
PU_API void pu_dpsk_destroy(pu_dpsk* h);
PU_API int pu_dpsk_bits_per_symbol(const pu_dpsk* h);
/* B frames of L samples; data symbols start at sample data_start of every frame.
 *   ref_mode 0: differential reference (1,0), a fresh / reset() demodulator (:881-886);
 *   ref_mode 1: setReferenceSymbol on the symbol that ends at data_start (:889-892; what findPreamble does, :470-478);
 *   est_cfo_hz[B] / phase_offset[B]: the members estimated_cfo_ / initial_phase_offset_ that findPreamble or
 *   setReferenceWithTraining leave behind and demodulateSoft compensates (:857-865); NULL = 0.
 * llr_out[b*llr_stride ...] = demodulateSoft() of the frame (:827-879), truncated to llr_stride floats. */
PU_API pu_status pu_dpsk_demod_soft_batch(pu_dpsk* h, const float* samples, size_t B, size_t L, size_t data_start,
                                          int ref_mode, const float* est_cfo_hz, const float* phase_offset,
                                          float* llr_out, size_t llr_stride, pu_memspace space, void* stream);
/* DPSKModulator (dpsk.hpp:102-307), host: layout 0 = generatePreamble() (Barker-13 x 3) + modulate(data), the frame of
 * tools/test_dpsk_snr.cpp:47-52; 1 = generateReferenceSymbol() + modulate; 2 = modulate only.  *out_len is always set. */
/* DPSKDemodulator::findPreamble (Barker-13 x 3 acquisition, dpsk.hpp:338-481, with computeDifferentialScore,
 * estimateCFOTolerant, refineTimingWithMatchedFilter and estimateInitialPhaseOffset) followed, when llr_out is not NULL, by
 * demodulateSoft on the span that starts at the returned data start -- the receive sequence of tools/test_dpsk_snr.cpp:66-73
 * for B frames.  data_start[B] = findPreamble's return value (-1: no preamble), est_cfo_hz[B] / phase_offset[B] = the members it
 * leaves behind, n_llr[B] = soft bits written to llr_out[b*llr_stride ...] (capped at llr_stride; rows are not cleared).
 * PU_ERR_UNSUPPORTED for samples_per_symbol > 512. */
PU_API pu_status pu_dpsk_receive_batch(pu_dpsk* h, const float* samples, size_t B, size_t L, float* llr_out, size_t llr_stride,
                                       int32_t* n_llr, int32_t* data_start, float* est_cfo_hz, float* phase_offset,
                                       pu_memspace space, void* stream);
PU_API pu_status pu_dpsk_tx(const pu_dpsk_config* cfg, int layout, const uint8_t* data, size_t n_bytes, float* out,
                            size_t out_cap, size_t* out_len);
/* Batched transmitter on the GPU (SURVEY 8f next-3): LDPCEncoder::encode of one block (payload zero-padded to k bits) followed by
 * DPSKModulator::generatePreamble() + modulate() (dpsk.hpp:118-153,212-279) for B payloads at once, i.e. the frame of
 * tools/test_dpsk_snr.cpp:40-60 with a fresh payload per trial; peak > 0 rescales every frame to that peak amplitude.  `code`
 * supplies the code rate.  out[B][out_stride] receives *frame_len samples per row; B = 0 queries *frame_len.  Waveforms are
 * bit-identical to pu_ldpc_encode + pu_dpsk_tx(layout 0). */
PU_API pu_status pu_dpsk_tx_batch(pu_dpsk* h, const pu_ldpc* code, const uint8_t* payload, size_t payload_stride, size_t payload_bytes,
                                  size_t B, float peak, float* out, size_t out_stride, size_t* frame_len, pu_memspace space, void* stream);

/* ---------------------------------------------------------------- multi-carrier DPSK (externally timed)
 * Replaces ultra::MultiCarrierDPSKDemodulator (src/psk/multi_carrier_dpsk.hpp:258-701) on frames that start at the
 * training sequence: [training_symbols][1 reference symbol][data symbols] -- what processGotChirp (:533-627) sees
 * after an external chirp detection.  POD mirror of MultiCarrierDPSKConfig (:26-89). */
typedef struct {
    float sample_rate;            /* 48000 */
    float freq_low, freq_high;    /* 500, 2500 */
    uint32_t num_carriers;        /* 3..20 */
    uint32_t samples_per_symbol;  /* 512 */
    uint32_t bits_per_symbol;     /* 2 DQPSK, 1 DBPSK */
    uint32_t training_symbols;    /* 8 */
} pu_mcdpsk_config;
typedef struct pu_mcdpsk pu_mcdpsk;
PU_API pu_status pu_mcdpsk_create(pu_ctx* ctx, const pu_mcdpsk_config* cfg, pu_mcdpsk** out);
PU_API void pu_mcdpsk_destroy(pu_mcdpsk* h);
/* setReference (:424-435) + demodulateSoft (:437-472) per frame; residual_cfo_hz[B] (may be NULL) receives cfo_hz_
 * after processTraining (:390-422) so the caller can apply the |cfo| > 5 Hz rejection of :591-598.  The CFO
 * correction through the 127-tap Hilbert FIR (:633-658) only runs for |cfo| > 0.1 Hz and is not part of this path. */
PU_API pu_status pu_mcdpsk_demod_soft_batch(pu_mcdpsk* h, const float* samples, size_t B, size_t L, float* llr_out,
                                            size_t llr_stride, float* residual_cfo_hz, pu_memspace space, void* stream);
/* MultiCarrierDPSKDemodulator behind an externally detected chirp, as MCDPSKWaveform::process drives it
 * (src/waveform/mc_dpsk_waveform.cpp:144-170: setChirpDetected(cfo) -> process(training + ref + data) -> getSoftBits), i.e.
 * processGotChirp (multi_carrier_dpsk.hpp:533-627): the frame is first frequency-shifted through the 127-tap Hilbert FIR when
 * |chirp_cfo_hz[b]| > 0.1 Hz (applyCFOCorrection :633-658), then processTraining / the 5 Hz false-positive rule / setReference /
 * demodulateSoft.  n_llr[B] = soft bits handed out (0 for a rejected or too short frame), cfo_after_hz[B] = getEstimatedCFO(). */
PU_API pu_status pu_mcdpsk_got_chirp_batch(pu_mcdpsk* h, const float* samples, size_t B, size_t L, const float* chirp_cfo_hz,
                                           float* llr_out, size_t llr_stride, int32_t* n_llr, float* cfo_after_hz,
                                           pu_memspace space, void* stream);
/* The IWaveform receive sequence of tools/test_iwaveform.cpp:127-160 on MC-DPSK frames [up chirp][gap][down chirp][gap][training]
 * [reference][data], for B frames: MCDPSKWaveform::detectSync (src/waveform/mc_dpsk_waveform.cpp:100-142: ChirpSync::detectDualChirp,
 * start_sample = up_chirp_start + 2 chirps + 2 gaps) -> setFrequencyOffset(cfo) (:71-76) -> process(span from start_sample)
 * (:144-170, i.e. pu_mcdpsk_got_chirp_batch on the located span) -> getSoftBits.
 *   sync_info[B][4]   = {detected, up_chirp_start, down_chirp_start, SyncResult::start_sample (training start) or -1}
 *   sync_values[B][4] = {cfo_hz, up correlation, down correlation, 0}
 *   llr_out[B][llr_stride] (may be NULL: detection only, i.e. IWaveform::detectSync; n_llr and cfo_after_hz are then unused),
 *   n_llr[B] = soft bits handed out (0: no chirp, start beyond the buffer, too short, or rejected by the 5 Hz rule); entries of
 *   llr_out[b] beyond n_llr[b] are unspecified; cfo_after_hz[B] = estimatedCFO(); threshold <= 0 selects the callers' 0.15. */
PU_API pu_status pu_mcdpsk_chirp_receive_batch(pu_mcdpsk* h, const float* samples, size_t B, size_t L, float threshold,
                                               float* llr_out, size_t llr_stride, int32_t* n_llr, int32_t* sync_info,
                                               float* sync_values, float* cfo_after_hz, pu_memspace space, void* stream);
/* MultiCarrierDPSKModulator (:91-257), host: generateTrainingSequence + generateReferenceSymbol + modulate(data). */
PU_API pu_status pu_mcdpsk_tx(const pu_mcdpsk_config* cfg, const uint8_t* data, size_t n_bytes, float* out, size_t out_cap,
                              size_t* out_len);
/* The same on the GPU for B payloads: LDPCEncoder::encode + generateTrainingSequence + generateReferenceSymbol + modulate
 * (multi_carrier_dpsk.hpp:118-243); bit-identical to pu_ldpc_encode + pu_mcdpsk_tx.  Arguments as pu_dpsk_tx_batch. */
PU_API pu_status pu_mcdpsk_tx_batch(pu_mcdpsk* h, const pu_ldpc* code, const uint8_t* payload, size_t payload_stride, size_t payload_bytes,
                                    size_t B, float peak, float* out, size_t out_stride, size_t* frame_len, pu_memspace space, void* stream);
/* As pu_ofdm_set_tx_interleave for pu_mcdpsk_tx_batch: the 648 coded bits are interleaved before the differential encoding; the zero
 * padding of the last symbol is unchanged.  0 (the default) switches it off.  Deinterleave with pu_llr_deinterleave_batch. */
PU_API pu_status pu_mcdpsk_set_tx_interleave(pu_mcdpsk* h, size_t bits_per_symbol);

/* ---------------------------------------------------------------- channel simulator
 * Replaces sim::WattersonChannel (src/sim/hf_channel.hpp:34-299) for batches of frames.  POD mirror of
 * WattersonChannel::Config (:36-65); the CFO injector fields (cfo_hz) are a separate call, pu_channel_apply_cfo_batch. */
typedef struct {
    float delay_spread_ms;      /* second path delay; effective delay is floor(ms*fs/1000)+1 samples (Q11) */
    float doppler_spread_hz;
    float path1_gain, path2_gain;
    uint32_t sample_rate;
    uint32_t fading_enabled, multipath_enabled, noise_enabled;
} pu_channel_config;
/* Derived constants of a config (delay d, IIR coefficient a, sqrt(1/a), the scan multipliers (1-a)^(4 2^s) for s < 5 and the
 * carry weights (1-a)^(4 l) for l < 32): the numbers the CPU twin needs to regenerate a frame bit for bit.  Any output pointer
 * may be NULL. */
PU_API pu_status pu_channel_params(const pu_channel_config* cfg, int32_t* delay_samples, float* alpha,
                                   float* noise_scale, float* apow2_5, float* apl_32);
/* Noise standard deviation for one TX waveform (host): convention 0 = WattersonChannel::process, rms(input) *
 * 10^(-snr/20) (hf_channel.hpp:110-119); convention 1 = the AWGN tools, sqrt(mean power / 10^(snr/10))
 * (tools/test_mode_snr.cpp:58-61). */
PU_API float pu_channel_noise_std(const float* tx, size_t L, float snr_db, int convention);
/* The same for every row of tx[B][tx_stride] on the DEVICE (frames produced by pu_ofdm_tx_batch): snr_factor[b] =
 * powf(10, snr_db/10) (convention 1) or powf(10, -snr_db/20) (convention 0), evaluated by the caller on the host. */
PU_API pu_status pu_channel_noise_std_batch(pu_ctx* ctx, const float* tx, size_t tx_stride, size_t L, size_t B,
                                            const float* snr_factor, int convention, float* noise_std, void* stream);
/* rx[b] = channel(tx_pool[tx_index[b]]) for b < B: frames of L samples, per-frame noise_std and 64-bit seed.
 * The random stream is the counter-based generator specified in csrc/pu_rng.cuh (NOT the reference's
 * mt19937 stream): frame b is a pure function of (config, tx waveform, noise_std[b], seed[b]).
 * tx_index == NULL uses waveform 0 for every frame. */
PU_API pu_status pu_channel_apply_batch(pu_ctx* ctx, const pu_channel_config* cfg, const float* tx_pool,
                                        size_t pool_stride, size_t pool_count, const uint32_t* tx_index,
                                        const float* noise_std, const uint64_t* seed, size_t B, size_t L,
                                        float* rx, pu_memspace space, void* stream);

/* The CFO injector of the reference's tools (tools/test_iwaveform.cpp:67-118): analytic signal through FFT / inverse FFT over the next
 * power of two, rotation by the float phase recurrence, real part -- applied by the tools to the CLEAN transmit audio before the
 * channel (:501-506), which is where pu_linksim_run applies it (pu_sweep_mode.cfo_hz, once per TX pool waveform; fresh payloads take
 * pu_tools_cfo_apply_batch below).  Host function, in
 * place; arrays shorter than 128 samples or |cfo| < 0.001 Hz are left untouched.  Bit-identical to the tool. */
PU_API pu_status pu_tools_apply_cfo(float* samples, size_t n, float cfo_hz, float sample_rate);
/* The same injector on the GPU for a batch of rows (csrc/tools_cfo_gpu.cu): a handle per (n, cfo_hz, sample_rate) holds the twiddles,
 * the rotator of the phase recurrence (both built by the host function's own code) and 64 MiB of scratch.  apply_batch works in place
 * on samples[b*stride .. b*stride + n) for b < B; every sample is bit-identical to pu_tools_apply_cfo on that row, and the samples
 * between n and stride are not written.  For n < 128 or |cfo_hz| < 0.001 rows are untouched and nothing is launched.  n up to 2^20
 * (PU_ERR_UNSUPPORTED above; the host function has no such limit).  PU_MEM_DEVICE enqueues on `stream` and does not synchronise the
 * host; PU_MEM_HOST stages the rows through the device and returns when they are written back. */
typedef struct pu_tools_cfo pu_tools_cfo;
PU_API pu_status pu_tools_cfo_create(pu_ctx* ctx, size_t n, float cfo_hz, float sample_rate, pu_tools_cfo** out);
PU_API void pu_tools_cfo_destroy(pu_tools_cfo* h);
PU_API pu_status pu_tools_cfo_apply_batch(pu_tools_cfo* h, float* samples, size_t B, size_t stride, pu_memspace space, void* stream);

/* WattersonChannel::applyCFO (hf_channel.hpp:173-232), the channel's optional carrier-frequency-offset injector, applied IN PLACE to
 * every row of samples[B][stride] (L samples each) with cfo_hz[b] and a CFO phase of 0 at the start of the row: down-mix around
 * 1500 Hz, 48-tap running-sum lowpass, rotation, up-mix.  Rows with |cfo| <= 0.001 Hz or fewer than 256 samples are left untouched, as
 * in the reference.  Deterministic: bit-identical to the reference (no random draw is involved). */
PU_API pu_status pu_channel_apply_cfo_batch(pu_ctx* ctx, float* samples, size_t B, size_t L, size_t stride, const float* cfo_hz,
                                            uint32_t sample_rate, pu_memspace space, void* stream);

/* ---------------------------------------------------------------- receive + decode, error counting
 * One call per batch of frames = the body of the reference's Monte-Carlo trial loop after the channel
 * (tools/test_ofdm_chirp_pilots.cpp:225-260): processPresynced -> first 648 soft bits -> decodeSoft.
 * LLRs never leave the device.  Frames that yield fewer than 648 soft bits are decoded with the missing
 * LLRs as erasures (0), like LDPCDecoder::decodeSoft's zero padding (ldpc_decoder.cpp:160-166). */
PU_API pu_status pu_receive_decode_batch(pu_ofdm* ofdm, pu_ldpc* ldpc, const float* samples, size_t B, size_t L,
                                         int training_symbols, const float* cfo_hz, const float* cfo_phase,
                                         uint8_t* info_bytes, size_t info_stride, uint8_t* ok, int32_t* iters,
                                         pu_memspace space, void* stream);
/* ---------------------------------------------------------------- protocol-v2 multi-codeword frames (SURVEY 8f next-4)
 * RxPipeline::decodeFrame(soft_bits, num_codewords) (src/gui/modem/rx_pipeline.cpp:348-445) for B frames, all codewords at the
 * decoder handle's rate (the rule of :356-365): decode CW0 (v2::decodeSingleCodeword, src/protocol/frame_v2.cpp:1134-1156) ->
 * parseHeader (:1175-1230: magic 0x554C, control/data layout, CRC-16) -> expected = TOTAL_CW -> "waiting" when num_codewords <
 * expected -> decode CW1+ -> success iff all decoded -> CodewordStatus::reassemble (:952-982,1023-1044: CW1+ lose their 0xD5/index
 * prefix).  llr[B][num_codewords][648]; frame_out[B][frame_cap] (bytes beyond frame_cap are dropped), frame_len[B] = size of
 * RxFrameResult::frame_data (0 unless success); info[B][5] = {success, frame_type, codewords_ok, codewords_failed, expected
 * codewords (0 = CW0 failed or header invalid)}.  One launch of the LDPC kernel over all B*num_codewords codewords + one assembly
 * kernel.  A data header with TOTAL_CW = 0 is undefined in the reference (out-of-bounds write); here: success, empty frame. */
PU_API pu_status pu_frame_decode_batch(pu_ctx* ctx, pu_ldpc* dec, const float* llr, size_t B, size_t num_codewords,
                                       uint8_t* frame_out, size_t frame_cap, int32_t* frame_len, int32_t* info,
                                       pu_memspace space, void* stream);
/* v2::encodeFrameWithLDPC(frame_data, rate) (frame_v2.cpp:1079-1127), host: out = n_codewords x 81 bytes; out == NULL queries
 * the codeword count. */
PU_API pu_status pu_frame_encode(int code_rate, const uint8_t* frame, size_t n_bytes, uint8_t* out, size_t out_cap,
                                 size_t* n_codewords);
/* LDPCEncoder::encode of one block per row on the GPU: payload[b * payload_stride ..+ payload_bytes) (payload_bytes <= k / 8, zero padded
 * to k bits) -> coded[b * coded_stride ..+ 81).  Bit-identical to pu_ldpc_encode.  One CTA per row, the encoder of pu_ofdm_tx_batch.
 * PU_MEM_HOST stages through the context; bytes beyond 81 in a row are not written. */
PU_API pu_status pu_ldpc_encode_batch(const pu_ldpc* code, const uint8_t* payload, size_t payload_stride, size_t payload_bytes, size_t B,
                                      uint8_t* coded, size_t coded_stride, pu_memspace space, void* stream);
/* v2::encodeFrameWithLDPC (frame_v2.cpp:1079-1127) per row on the GPU at the code's rate: frames[b * frame_stride ..+ frame_bytes) ->
 * coded[b * coded_stride ..+ n_codewords * 81).  Bit-identical to pu_frame_encode; at most 255 codewords, as pu_frame_tx_batch (whose
 * encoder it is).  B == 0 or coded == NULL only sets *n_codewords.  Bytes beyond n_codewords * 81 in a row are not written. */
PU_API pu_status pu_frame_encode_batch(const pu_ldpc* code, const uint8_t* frames, size_t frame_stride, size_t frame_bytes, size_t B,
                                       uint8_t* coded, size_t coded_stride, size_t* n_codewords, pu_memspace space, void* stream);

/* Frame-error rule of the tools (tools/test_mode_snr.cpp:98-104): success iff lastDecodeSuccess() and the first
 * payload_bytes decoded bytes equal the payload.  DEVICE pointers.  counters[bin[b]][6] (uint64, atomically
 * accumulated) = {frames, frame_errors, bit_errors, payload_bits, decode_failures, iteration_sum};
 * tx_index selects the payload row, bin the counter row (NULL = row 0). */
PU_API pu_status pu_count_errors(pu_ctx* ctx, const uint8_t* info_bytes, size_t info_stride, const uint8_t* ok,
                                 const int32_t* iters, const uint8_t* payload_pool, size_t payload_stride,
                                 const uint32_t* tx_index, const uint32_t* bin, size_t payload_bytes, size_t B,
                                 uint64_t* counters, void* stream);
/* Pre-decoder (raw) bit errors: soft bits against the coded bits sent, DEVICE pointers.  For b < B and j < n_bits, soft bit
 * llr[b * llr_stride + j] (decoder order, i.e. after any deinterleaving) against bit j (MSB first) of coded[coded_index[b] *
 * coded_stride ...] (coded_index NULL = row b).  Positions j >= n_valid[b] (n_valid NULL = all valid) and soft bits equal to +-0 are
 * erasures; otherwise the hard decision is 1 iff llr < 0 (the decoder's rule).  counters[bin[b]][4] (uint64, accumulated with integer
 * atomics, so a table does not depend on the launch order) = {soft_bits (n_bits per row), erasures, bit_errors (erasures excluded),
 * strong_errors (bit errors with |llr| >= strong)}; bin NULL = row 0.  The sweep passes strong = 10, the clipLLR bound of the OFDM
 * demappers and the clamp of the MC-DPSK demapper; single-carrier DPSK soft bits stop at 5, so that column is 0 for its rows (and
 * MC-DPSK's errors were not seen to reach 10 in the reduced sweep table either). */
PU_API pu_status pu_count_raw_errors(pu_ctx* ctx, const float* llr, size_t llr_stride, size_t n_bits, const int32_t* n_valid,
                                     const uint8_t* coded, size_t coded_stride, const uint32_t* coded_index, const uint32_t* bin,
                                     size_t B, float strong, uint64_t* counters, void* stream);

/* ---------------------------------------------------------------- Monte-Carlo sweep driver (BASELINE.json config 5)
 * The reference runs its FER/BER waterfalls as a shell matrix over one-process-per-cell tools (tests/regression_matrix.sh:139-243 over
 * the loop of tools/test_iwaveform.cpp:597-806 and tools/test_mode_snr.cpp:40-105: per trial  payload -> encode -> modulate -> channel
 * -> sync/demodulate -> decodeSoft -> compare).  pu_linksim_run is that matrix as ONE call per GPU rank: a mode table (waveform x
 * modulation x code rate x channel) x an SNR grid x trials_per_point seeds is cut into work units (mode, SNR point, seed block), the
 * units are dealt to the ranks by expected cost (longest-processing-time first: low-SNR blocks run more LDPC iterations, acquisition
 * modes cost orders of magnitude more per frame), and every rank runs its units in large mixed-SNR batches through
 * pu_channel_apply_batch -> the waveform's receive entry point -> pu_ldpc_decode_batch -> pu_count_errors.  Frames are pure functions
 * of (mode, SNR index, trial): seed = base_seed << 40 ^ mode << 56 ^ snr_index << 32 ^ trial, TX waveform = trial % pool; no data is
 * exchanged between ranks, the counter tables are summed once at the end (pu_counters_allreduce, or the host's own collective).
 * With manifest_dir set every finished unit is appended to a per-rank shard file; a later call with the same table resumes: finished
 * units (from ANY earlier world size) are skipped and their counters are returned by rank 0. */
enum { PU_WF_OFDM = 0,           /* 2 LTS + data, genie timing: processPresynced (tools/test_ofdm_chirp_pilots.cpp:183-260) */
       PU_WF_OFDM_SC = 1,        /* Schmidl-Cox preamble + data fed to process() in chunks (tools/test_mode_snr.cpp:40-105) */
       PU_WF_OFDM_CHIRP = 2,     /* dual chirp + training + data: detectSync -> setFrequencyOffset -> process (tools/test_iwaveform.cpp:127-160) */
       PU_WF_DPSK = 3,           /* Barker preamble + data, genie data start (setReferenceSymbol on the last preamble symbol) */
       PU_WF_DPSK_ACQ = 4,       /* ... received through findPreamble (tools/test_dpsk_snr.cpp:66-73) */
       PU_WF_MCDPSK = 5,         /* training + reference + data, externally timed (tools/test_mc_dpsk.cpp:180-196) */
       PU_WF_MCDPSK_CHIRP = 6 }; /* dual chirp + training + reference + data through MCDPSKWaveform's detectSync / process */
/* channel presets: ccir:: (src/sim/hf_channel.hpp:305-381) and itu_r_f1487:: (:402-487) */
enum { PU_CH_AWGN = 0, PU_CH_GOOD = 1, PU_CH_MODERATE = 2, PU_CH_POOR = 3, PU_CH_FLUTTER = 4,
       PU_CH_ITU_GOOD = 5, PU_CH_ITU_MODERATE = 6, PU_CH_ITU_POOR = 7, PU_CH_ITU_FLUTTER = 8 };
PU_API pu_status pu_channel_preset(int preset, pu_channel_config* out);

typedef struct {
    uint32_t waveform;          /* PU_WF_* */
    pu_modem_config ofdm;       /* PU_WF_OFDM*  */
    pu_dpsk_config dpsk;        /* PU_WF_DPSK*  */
    pu_mcdpsk_config mcdpsk;    /* PU_WF_MCDPSK* */
    uint32_t code_rate;         /* PU_RATE_* */
    uint32_t payload_bytes;     /* compared bytes (<= k/8) */
    uint32_t channel;           /* PU_CH_* */
    uint32_t n_snr;
    float snr_first_db, snr_step_db;
    float peak;                 /* > 0: the tools' peak normalisation of every TX waveform (tools/test_mode_snr.cpp:54-56) */
    uint32_t precision;         /* pu_precision of the OFDM kernels */
    uint32_t chunk;             /* PU_WF_OFDM_SC: process() chunk, 0 = 960 */
    float cost;                 /* relative cost of one frame for the partitioner; 0 = built-in estimate */
    uint32_t lead_samples;      /* silence in front of / behind every TX waveform (tools/test_iwaveform.cpp:396-459 surrounds its frames with */
    uint32_t tail_samples;      /* 1.5 s / 1 s of it): an acquired frame whose tail the channel's delay pushes out of the buffer loses its last symbol */
    float cfo_hz;               /* the tools' --cfo: pu_tools_apply_cfo on every TX waveform (silence included) before the channel; 0 = none */
    uint32_t fresh_payloads;    /* 1: a new payload per trial, encoded and modulated on the GPU (pu_*_tx_batch) inside the batch, as the tools do
                                 * (tools/test_dpsk_snr.cpp:40-60, tools/test_mode_snr.cpp:40-60), instead of the pool of TX waveforms; the
                                 * payload is a pure function of (base_seed, mode, SNR index, trial).  Each row is built in the pool's order: body
                                 * behind the lead silence and the chirp pair, peak normalisation over chirp and body, cfo_hz through
                                 * pu_tools_cfo_apply_batch over the whole row, then the row's noise level. */
    uint32_t frame_payload_bytes; /* > 0: every trial is a protocol-v2 DATA frame with this many payload bytes (several codewords in one
                                 * OFDM frame; PU_WF_OFDM, PU_WF_OFDM_SC and PU_WF_OFDM_CHIRP only, at most 65535 bytes and 255 codewords)
                                 * and the counters of its SNR points are whole-frame counters {frames, frame_errors, codewords_failed,
                                 * codewords sent, header_failures, 0}: a frame is lost unless RxPipeline::decodeFrame (rx_pipeline.cpp:
                                 * 348-445) returns exactly the frame sent.  The frame is DataFrame::serialize of {type 0x30, flags 0x01,
                                 * src 0x123456, dst 0xABCDEF}: pool waveform i carries pu_sweep_payload(base_seed, mode, i) with seq i + 1,
                                 * a fresh frame the fresh payload bytes with seq = trial & 0xFFFF.  Acquired frames deliver
                                 * min(n_cw, soft bits / 648) codewords to the decoder.  payload_bytes is unused (0 allowed); 0 = codeword mode */
    uint32_t interleave_bps;    /* > 0: ChannelInterleaver(interleave_bps, 648) on every codeword, as the reference's IWaveform path does
                                 * (getSoftBits -> ChannelInterleaver::deinterleave -> decodeSoft): the pool interleaves each codeword's bytes
                                 * before modulating them, fresh frames through pu_*_set_tx_interleave; the receiver deinterleaves
                                 * (PU_WF_OFDM codewords: pu_ofdm_set_deinterleave, fused; everything else: pu_llr_deinterleave_batch on
                                 * every codeword).  OFDM and MC-DPSK waveforms, codeword and frame modes; a nonzero value on PU_WF_DPSK /
                                 * PU_WF_DPSK_ACQ makes the table invalid.  0 = no interleaving */
} pu_sweep_mode;

typedef struct {
    const pu_sweep_mode* modes;
    uint32_t n_modes;
    uint32_t pool;              /* TX waveforms per mode (0 = 64); payload of waveform i = pu_sweep_payload(base_seed, mode, i) */
    uint64_t trials_per_point;  /* seeds per (mode, SNR point) */
    uint32_t block_trials;      /* trials per work unit (0 = 4096) */
    uint32_t max_iter;          /* LDPC iteration limit (0 = 50) */
    uint64_t base_seed;         /* 16 bits used (0 = 0xB200) */
    uint32_t rank, world;
    uint64_t batch_bytes;       /* device memory for one batch of channel outputs (0 = 1.5 GiB) */
    const char* manifest_dir;   /* NULL = no persistence / resume */
    uint64_t max_units;         /* stop after this many units on this rank (0 = run everything): tests of resume */
    uint64_t run_id;            /* manifest only: equal on all ranks of one launch, different between launches (e.g. the launch time).
                                 * Shards written under the current run_id are ignored when the finished set is read, so a rank that
                                 * starts late sees the same finished units -- hence computes the same partition -- as its peers */
} pu_sweep_desc;

typedef struct {
    uint64_t units_total, units_resumed, units_run, frames_run;
    double seconds;             /* wall time of the run loop on this rank */
    double setup_seconds;       /* ... of which building the modes' TX pools, noise tables and handles on the host, */
    double wait_seconds;        /* ... blocked on the GPU (batch k-2 not finished when batch k is due): GPU-bound share, */
    double fill_seconds;        /* ... writing batch descriptors on the host, */
    double enqueue_seconds;     /* ... inside the C-ABI calls that enqueue a batch (copies + kernel launches) */
    double busy_cost, total_cost; /* this rank's share / the sum of the partitioner's cost estimates (remaining units) */
} pu_sweep_stats;

/* number of work units of a table, and the offset of mode m's SNR point 0 in the counter table (= sum of n_snr of the modes before) */
PU_API uint64_t pu_sweep_unit_count(const pu_sweep_desc* d);
PU_API uint32_t pu_sweep_point_count(const pu_sweep_desc* d);
/* owner[u] = rank that runs unit u (0xffffffff for units marked in done[u] != 0; done may be NULL); cost[u] may be NULL.
 * Pure host function of the table: every rank computes the same assignment. */
PU_API pu_status pu_sweep_partition(const pu_sweep_desc* d, const uint8_t* done, uint32_t* owner, double* cost);
/* unit u -> (mode, SNR index, first trial, number of trials) */
PU_API pu_status pu_sweep_unit(const pu_sweep_desc* d, uint64_t u, uint32_t* mode, uint32_t* snr_index, uint64_t* first_trial, uint32_t* n_trials);
/* payload bytes of TX waveform `index` of mode `mode` (splitmix64 stream; lets any host regenerate the pool) */
PU_API void pu_sweep_payload(uint64_t base_seed, uint32_t mode, uint32_t index, uint8_t* out, size_t n_bytes);
/* counters[pu_sweep_point_count][6] (HOST, uint64) = this rank's {frames, frame_errors, bit_errors, payload_bits, decode_failures,
 * iteration_sum} per (mode, SNR point) -- whole-frame counters for frame modes (pu_sweep_mode.frame_payload_bytes) --, rank 0
 * additionally holding the resumed units; stats may be NULL. */
PU_API pu_status pu_linksim_run(pu_ctx* ctx, const pu_sweep_desc* d, uint64_t* counters, pu_sweep_stats* stats);
/* pu_linksim_run with a second table: raw[pu_sweep_point_count][4] (HOST, uint64) = the pu_count_raw_errors counters {soft_bits, erasures,
 * bit_errors, strong_errors} (strong = 10) over every soft bit the decoder is given (648 per codeword trial, n_cw x 648 per frame trial;
 * the soft bits an acquiring receiver did not deliver are erasures, located through the deinterleaver's permutation when the mode
 * interleaves), or raw == NULL = exactly pu_linksim_run.  counters is the same table
 * pu_linksim_run returns: PU_WF_OFDM codewords leave the fused demodulate + decode call for its two halves, which decode the same.  A raw
 * run keys its manifest apart from a plain run of the same table (neither resumes from the other's shards) and records the 4 raw
 * counters of every unit behind its 6 counters; rank 0 returns the resumed raw counters too. */
PU_API pu_status pu_linksim_run_raw(pu_ctx* ctx, const pu_sweep_desc* d, uint64_t* counters, uint64_t* raw, pu_sweep_stats* stats);
/* Sum n uint64 counters over the ranks of an NCCL communicator (ncclComm_t passed as void*; libnccl is resolved at run time with
 * dlopen, the library does not link it).  PU_MEM_HOST stages through the context; comm == NULL is a no-op (single rank). */
PU_API pu_status pu_counters_allreduce(pu_ctx* ctx, uint64_t* counters, size_t n, void* nccl_comm, pu_memspace space, void* stream);
/* Wilson score interval of an error rate (the Monte-Carlo confidence interval of BASELINE.json's north star) */
PU_API void pu_wilson_interval(uint64_t errors, uint64_t n, double z, double* lo, double* hi);

/* ---------------------------------------------------------------- numerics pinning (tests)
 * Evaluates the device restatements of the host libm routines the reference's path calls (csrc/ref_math.cuh):
 * op 0 atan2f(a,b), 1 sinf(a), 2 cosf(a), 3 hypotf(a,b), 4 atanf(a).  ctx == NULL evaluates the same source on
 * the HOST (so it can be compared with libm without a GPU); otherwise on the device.  Host pointers. */
PU_API pu_status pu_refmath_eval(pu_ctx* ctx, int op, const float* a, const float* b, float* out, size_t n);

#ifdef __cplusplus
}
#endif
#endif /* PU_CAPI_H */
