"""Host side of the batched Monte-Carlo link simulation: TX waveform pool, channel, receive+decode, error
counters, sharding over ranks.  Everything heavy happens in libpu_b200.so through the C ABI (capi); torch is
used for device memory, streams and the one collective (all-reduce of the counter table).

Mirrors the reference's Monte-Carlo tools (tools/test_mode_snr.cpp:18-109, tools/test_ofdm_chirp_pilots.cpp:
100-270): per trial  encode -> modulate -> channel -> processPresynced -> getSoftBits -> decodeSoft -> compare.
"""
import ctypes as C
import math

import numpy as np

from . import capi

COUNTER_NAMES = ("frames", "frame_errors", "bit_errors", "bits", "decode_failures", "iteration_sum")
# pre-decoder counters of the soft bits the decoder is given (capi.count_raw_errors, pu_linksim_run_raw): soft bits, erasures (+-0, or not
# delivered by an acquiring receiver), hard-decision errors among the rest, and those of them with |llr| >= RAW_STRONG
RAW_COUNTER_NAMES = ("soft_bits", "erasures", "bit_errors", "strong_errors")
RAW_STRONG = 10.0          # the clipLLR bound of the OFDM demappers and the clamp of the MC-DPSK demapper


class ChannelConfig(C.Structure):
    """pu_channel_config: POD mirror of sim::WattersonChannel::Config (src/sim/hf_channel.hpp:36-65)."""
    _fields_ = [("delay_spread_ms", C.c_float), ("doppler_spread_hz", C.c_float), ("path1_gain", C.c_float),
                ("path2_gain", C.c_float), ("sample_rate", C.c_uint32), ("fading_enabled", C.c_uint32),
                ("multipath_enabled", C.c_uint32), ("noise_enabled", C.c_uint32)]


def channel_preset(name):
    """ccir:: presets of src/sim/hf_channel.hpp:305-381."""
    table = {"awgn": (0.0, 0.0, 1.0, 0.0, 0, 0), "good": (0.5, 0.1, 0.707, 0.707, 1, 1),
             "moderate": (1.0, 0.5, 0.707, 0.707, 1, 1), "poor": (2.0, 1.0, 0.707, 0.707, 1, 1),
             "flutter": (0.5, 10.0, 0.707, 0.707, 1, 1)}
    d, f, g1, g2, fad, mp = table[name]
    return ChannelConfig(d, f, g1, g2, 48000, fad, mp, 1)


def ofdm_tx(cfg, data, layout=0):
    """pu_ofdm_tx: OFDMModulator training/preamble + modulate on the host."""
    d = np.ascontiguousarray(data, dtype=np.uint8)
    n = C.c_size_t(0)
    capi.lib().pu_ofdm_tx(C.byref(cfg), int(layout), capi._ptr(d), C.c_size_t(len(d)), None, C.c_size_t(0), C.byref(n))
    out = np.zeros(n.value, np.float32)
    capi.check(capi.lib().pu_ofdm_tx(C.byref(cfg), int(layout), capi._ptr(d), C.c_size_t(len(d)), capi._ptr(out),
                                     C.c_size_t(len(out)), C.byref(n)))
    return out


def channel_noise_std(tx, snr_db, convention=0):
    f = capi.lib().pu_channel_noise_std
    f.restype = C.c_float
    x = np.ascontiguousarray(tx, dtype=np.float32)
    return float(f(capi._ptr(x), C.c_size_t(len(x)), C.c_float(snr_db), int(convention)))


def channel_apply(ctx, ch, tx_pool, tx_index, noise_std, seed, rx=None):
    """pu_channel_apply_batch.  numpy => host staging, torch.cuda => device."""
    tor = capi._is_torch(tx_pool)
    P, L = tx_pool.shape
    B = len(noise_std)
    if rx is None:
        if tor:
            import torch
            rx = torch.empty((B, L), dtype=torch.float32, device=tx_pool.device)
        else:
            rx = np.zeros((B, L), np.float32)
    sp = capi._space(tx_pool, tx_index, noise_std, seed, rx)
    capi.check(capi.lib().pu_channel_apply_batch(ctx._h, C.byref(ch), capi._ptr(tx_pool), C.c_size_t(L), C.c_size_t(P),
                                                 capi._ptr(tx_index), capi._ptr(noise_std), capi._ptr(seed),
                                                 C.c_size_t(B), C.c_size_t(L), capi._ptr(rx), sp, capi._stream(sp)))
    return rx


def channel_apply_cfo(ctx, rx, cfo_hz, sample_rate=48000):
    """pu_channel_apply_cfo_batch: WattersonChannel::applyCFO in place on every row of rx [B, L] (numpy => host, torch.cuda => device)."""
    B, L = rx.shape
    sp = capi._space(rx, cfo_hz)
    stride = rx.stride(0) if capi._is_torch(rx) else L
    capi.check(capi.lib().pu_channel_apply_cfo_batch(ctx._h, capi._ptr(rx), C.c_size_t(B), C.c_size_t(L), C.c_size_t(stride), capi._ptr(cfo_hz),
                                                     C.c_uint32(sample_rate), sp, capi._stream(sp)))
    return rx


def receive_decode(ofdm, ldpc, samples, training=2, cfo_hz=None, cfo_phase=None, info=None, ok=None, iters=None):
    """pu_receive_decode_batch: demodulate + LDPC decode; LLRs stay on the device."""
    tor = capi._is_torch(samples)
    B, L = samples.shape
    kb = ldpc.info_bytes
    if tor:
        import torch
        info = torch.empty((B, kb), dtype=torch.uint8, device=samples.device) if info is None else info
        ok = torch.empty(B, dtype=torch.uint8, device=samples.device) if ok is None else ok
        iters = torch.empty(B, dtype=torch.int32, device=samples.device) if iters is None else iters
    else:
        samples = np.ascontiguousarray(samples, dtype=np.float32)
        info = np.zeros((B, kb), np.uint8) if info is None else info
        ok = np.zeros(B, np.uint8) if ok is None else ok
        iters = np.zeros(B, np.int32) if iters is None else iters
    sp = capi._space(samples, info, ok, iters, cfo_hz, cfo_phase)
    capi.check(capi.lib().pu_receive_decode_batch(ofdm._h, ldpc._h, capi._ptr(samples), C.c_size_t(B), C.c_size_t(L),
                                                  int(training), capi._ptr(cfo_hz), capi._ptr(cfo_phase),
                                                  capi._ptr(info), C.c_size_t(kb), capi._ptr(ok), capi._ptr(iters),
                                                  sp, capi._stream(sp)))
    return info, ok, iters


def count_errors(ctx, info, ok, iters, payload_pool, tx_index, bins, payload_bytes, counters):
    """pu_count_errors on device tensors; counters is a torch.int64 [n_bins, 6] tensor accumulated in place."""
    import torch
    B = info.shape[0]
    capi.check(capi.lib().pu_count_errors(ctx._h, capi._ptr(info), C.c_size_t(info.stride(0)), capi._ptr(ok),
                                          capi._ptr(iters), capi._ptr(payload_pool), C.c_size_t(payload_pool.stride(0)),
                                          capi._ptr(tx_index), capi._ptr(bins), C.c_size_t(payload_bytes), C.c_size_t(B),
                                          capi._ptr(counters), C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return counters


def interleave_codewords(coded, bps):
    """ChannelInterleaver(bps, 648)::interleave (out[perm[i]] = in[i], bits MSB first) of every 81-byte codeword of `coded`, each on its own,
    as the reference's IWaveform transmitters do before modulating."""
    perm = capi.channel_interleaver_perm(bps)[0]
    bits = np.unpackbits(np.ascontiguousarray(coded, np.uint8).reshape(-1, 81), axis=1)
    out = np.zeros_like(bits)
    out[:, perm] = bits
    return np.packbits(out, axis=1).reshape(-1)


def erase_undelivered(llr, n_valid, n_bits, bps):
    """llr[:, :n_bits] (decoder order, behind ChannelInterleaver(bps, 648)::deinterleave of every codeword) with +0 at every soft bit the
    receiver did not deliver: n_valid[b] counts soft bits in the receiver's order, and decoder bit c * 648 + i came from its position
    c * 648 + perm[i] (out[perm[i]] = in[i] on the transmit side).  A copy; the decoder's input stays as it is."""
    import torch
    perm = torch.from_numpy(capi.channel_interleaver_perm(bps)[0].astype(np.int64)).to(llr.device)
    pos = (torch.arange(n_bits // 648, device=llr.device)[:, None] * 648 + perm[None, :]).reshape(-1)
    out = llr[:, :n_bits].clone()
    out[pos[None, :] >= n_valid.to(torch.int64)[:, None]] = 0.0
    return out


def count_raw(ctx, llr, coded, raw, n_bits, n_valid, index, bins, bps):
    """Raw counts of soft bits in decoder order; n_valid (None = all delivered) counts the soft bits the receiver delivered in ITS order,
    which a deinterleaver (bps > 0) permutes: the undelivered ones are then zeroed in a copy (erase_undelivered) before counting."""
    if n_valid is not None and bps:
        llr, n_valid = erase_undelivered(llr, n_valid, n_bits, bps), None
    capi.count_raw_errors(ctx, llr, coded, raw, n_bits, n_valid, index, bins, RAW_STRONG)


def wilson_interval(errors, n, z=1.96):
    """Wilson score interval for an error rate (the Monte-Carlo confidence interval of the north star)."""
    if n == 0:
        return 0.0, 1.0
    p = errors / n
    den = 1 + z * z / n
    mid = (p + z * z / (2 * n)) / den
    half = z * math.sqrt(p * (1 - p) / n + z * z / (4 * n * n)) / den
    return max(0.0, mid - half), min(1.0, mid + half)


class LinkSim:
    """One waveform mode x code rate x channel: owns the TX pool and runs sharded SNR sweeps on one GPU.

    cfg selects the waveform: capi.ModemConfig (OFDM, presynced frame = 2 LTS + data, tools/test_ofdm_chirp_pilots.cpp:
    183-191), capi.DpskConfig (single-carrier DPSK, Barker preamble + data, tools/test_dpsk_snr.cpp:47-52, genie data
    start) or capi.McDpskConfig (multi-carrier DPSK, training + reference + data, tools/test_mc_dpsk.cpp:180-196).
    peak=0.5 applies the tools' peak normalisation (tools/test_mode_snr.cpp:54-56).  tools_cfo_hz applies the tools' tuning error
    (tools/test_iwaveform.cpp:501-506) to every clean TX waveform after it: capi.tools_apply_cfo on the pool, capi.ToolsCfo on fresh frames.
    lead_samples / tail_samples (layout 'chirp') surround every frame with silence before both, as the tools do (test_iwaveform.cpp:396-459):
    a positive tuning error moves the up chirp's apparent start in front of the frame, so without a lead the chirp's timing is lost.
    interleave_bps > 0 (OFDM and MC-DPSK) passes every codeword through ChannelInterleaver(interleave_bps, 648) as the sweep driver does
    (pu_sweep_mode.interleave_bps): the pool interleaves the coded bytes, fresh frames the transmitter (set_tx_interleave); the presynced
    OFDM receiver deinterleaves in its LLR write (set_deinterleave), every other receiver through capi.llr_deinterleave_batch.

    Frames are identified by (snr index, trial index); frame -> (tx waveform, seed) is a pure function, so any
    frame can be regenerated, and ranks take disjoint trial ranges with no data exchange (SURVEY §8e).

    raw: an int64 [n_snr, 4] device tensor given to run_batch / receive_count accumulates RAW_COUNTER_NAMES of the soft bits the decoder
    gets against the coded bits sent (the pool's coded bytes before interleaving, or pu_ldpc_encode_batch of the fresh payloads), as
    pu_linksim_run_raw counts them; the presynced OFDM receiver then runs demodulator and decoder as two calls."""

    def __init__(self, ctx, cfg, channel="awgn", payload_bytes=40, pool=64, snr_convention=None, pool_seed=12345,
                 max_iter=50, device=None, code_rate=None, peak=None, layout="presynced", chunk=960, fresh_payload=False,
                 acquire=False, precision="exact", payloads=None, tools_cfo_hz=0.0,
                 lead_samples=0, tail_samples=0, interleave_bps=0):
        import torch
        self.ctx, self.cfg = ctx, cfg
        self.precision = precision
        self.device = device or torch.device("cuda", ctx.device)
        self.ch = channel_preset(channel) if isinstance(channel, str) else channel
        self.channel_name = channel if isinstance(channel, str) else "custom"
        # AWGN tools define SNR on mean frame power, WattersonChannel on input rms (same number, different rounding)
        self.snr_convention = (1 if self.channel_name == "awgn" else 0) if snr_convention is None else snr_convention
        if isinstance(cfg, capi.ModemConfig):
            self.kind = "ofdm"
            rate = cfg.code_rate if code_rate is None else code_rate
            self.ofdm = self.demod = capi.OfdmDemodulator(ctx, cfg)
            # "exact": FFT bins bit-identical to the reference; "fast": FMA butterflies, LLRs within 1e-4 (pu_ofdm_set_precision)
            self.ofdm.set_precision(precision)
            # layout "presynced": 2 LTS + data, genie timing (tools/test_ofdm_chirp_pilots.cpp); layout "sc": generatePreamble()
            # + data fed to process() in `chunk`-sample pieces, i.e. with Schmidl-Cox acquisition (tools/test_mode_snr.cpp:40-105)
            # layout "chirp": OFDM_CHIRP frames = ChirpSync::generate() + training + data, received through dual-chirp detectSync ->
            # setFrequencyOffset -> process (tools/test_iwaveform.cpp:127-160)
            assert layout in ("presynced", "sc", "chirp")
            self.layout, self.chunk = layout, chunk
            chirp = capi.chirp_generate(float(cfg.sample_rate), float(cfg.tx_cfo_hz)) if layout == "chirp" else None
            if layout == "chirp":
                build = lambda coded: np.concatenate([chirp, ofdm_tx(cfg, coded, 0)])
            else:
                build = lambda coded: ofdm_tx(cfg, coded, 1 if layout == "sc" else 0)
        elif isinstance(cfg, capi.DpskConfig):
            self.kind = "dpsk"
            rate = capi.R1_4 if code_rate is None else code_rate          # tools/test_dpsk_snr.cpp:28-29
            self.demod = capi.DpskDemodulator(ctx, cfg)
            self.data_start = 39 * cfg.samples_per_symbol                 # Barker-13 x 3 (dpsk.hpp:202-204)
            self.layout = "presynced"
            chirp = None
            build = lambda coded: capi.dpsk_tx(cfg, coded, 0)
        elif isinstance(cfg, capi.McDpskConfig):
            self.kind = "mcdpsk"
            rate = capi.R1_2 if code_rate is None else code_rate
            self.demod = capi.McDpskDemodulator(ctx, cfg)
            # layout "chirp": MC-DPSK frames as transmitted = ChirpSync::generate() + training + reference + data, received through
            # MCDPSKWaveform's detectSync -> setFrequencyOffset -> process (tools/test_iwaveform.cpp:127-160); a frame without chirp
            # or with fewer than 648 soft bits is lost
            assert layout in ("presynced", "chirp")
            self.layout = layout
            chirp = capi.chirp_generate(float(cfg.sample_rate), 0.0) if layout == "chirp" else None
            if layout == "chirp":
                build = lambda coded: np.concatenate([chirp, capi.mcdpsk_tx(cfg, coded)])
            else:
                build = lambda coded: capi.mcdpsk_tx(cfg, coded)
        else:
            raise TypeError("cfg must be a capi.ModemConfig, capi.DpskConfig or capi.McDpskConfig")
        self.code_rate = rate
        self.ldpc = capi.LdpcDecoder(ctx, rate, max_iter)
        # fresh_payload: every frame carries its own random payload, encoded and modulated on the GPU (pu_ofdm_tx_batch), as the
        # reference's tools do per trial (tools/test_mode_snr.cpp:44-56), instead of indexing a host-built pool of waveforms
        # acquire (single-carrier DPSK): Barker acquisition by findPreamble instead of genie timing, i.e. the receive sequence of
        # tools/test_dpsk_snr.cpp:66-73; a frame without preamble or with fewer than 648 soft bits is lost
        self.acquire = bool(acquire)
        assert not self.acquire or self.kind == "dpsk", "acquire=True is the DPSK Barker path; OFDM uses layout='sc'"
        self.fresh_payload = bool(fresh_payload)
        self.interleave_bps = int(interleave_bps)
        assert not self.interleave_bps or self.kind != "dpsk", "single-carrier DPSK has no ChannelInterleaver in the reference"
        if self.interleave_bps:
            self.demod.set_tx_interleave(self.interleave_bps)
            if self.kind == "ofdm" and self.layout == "presynced":
                self.ofdm.set_deinterleave(self.interleave_bps, 648)
        self.peak = peak
        self.chirp = None if chirp is None else torch.from_numpy(chirp).to(self.device)
        self.sample_rate = float(cfg.sample_rate)
        self.tools_cfo_hz = float(tools_cfo_hz)
        self.tools_cfo = None                  # capi.ToolsCfo of the fresh frames, made for their length on first use
        self.lead, self.tail = int(lead_samples), int(tail_samples)
        assert not (self.lead or self.tail) or self.layout == "chirp", "silence around a frame needs the acquiring receiver (layout='chirp')"
        self.payload_bytes = payload_bytes
        rng = np.random.default_rng(pool_seed)
        # payloads: explicit [pool, payload_bytes] array (e.g. the splitmix64 pool of the C++ sweep driver, capi.Sweep.payload)
        self.payloads = (rng.integers(0, 256, (pool, payload_bytes), dtype=np.uint8) if payloads is None
                         else np.ascontiguousarray(payloads, dtype=np.uint8).reshape(pool, payload_bytes))
        coded = [capi.ldpc_encode(rate, p) for p in self.payloads]
        self.coded_pool = torch.from_numpy(np.stack(coded)).to(self.device)      # [pool, 81], before interleaving: raw counts
        if self.interleave_bps:
            coded = [interleave_codewords(c, self.interleave_bps) for c in coded]
        waves = [np.pad(build(c), (self.lead, self.tail)) for c in coded]
        if peak is not None:
            waves = [(w * (np.float32(peak) / np.abs(w).max())).astype(np.float32) for w in waves]
        if self.tools_cfo_hz != 0.0:
            waves = [capi.tools_apply_cfo(w, self.tools_cfo_hz, self.sample_rate) for w in waves]
        self.L = len(waves[0])
        self.tx_host = np.stack(waves)
        self.tx_pool = torch.from_numpy(self.tx_host).to(self.device)
        kb = self.ldpc.info_bytes
        pad = np.zeros((pool, kb), np.uint8)
        pad[:, :payload_bytes] = self.payloads
        self.payload_pool = torch.from_numpy(pad).to(self.device)
        self.pool = pool

    def demod_llr(self, rx, llr=None):
        """First 648 soft bits of every frame (device tensors), as the tools consume them, in the decoder's order."""
        out = self._receiver_llr(rx, llr)
        if self.interleave_bps and not (self.kind == "ofdm" and self.layout == "presynced"):     # that one deinterleaves in its kernel
            capi.llr_deinterleave_batch(self.ctx, out, 1, self.interleave_bps)
        return out

    def _receiver_llr(self, rx, llr=None):
        if self.kind == "ofdm" and self.layout == "sc":
            out = self.demod.process_batch(rx, chunk=self.chunk, llr_stride=648)
            self.last_n_llr, self.last_sync = out[1], out[2]
            return out[0]
        if self.kind == "ofdm" and self.layout == "chirp":
            out = self.demod.chirp_receive_batch(rx, llr_stride=648)
            self.last_n_llr, self.last_sync = out[1], out[2]
            return out[0]
        if self.kind == "ofdm":
            return self.demod.presynced_batch(rx, 2, llr_stride=648, llr=llr, want_aux=False)[0]
        if self.kind == "dpsk" and self.acquire:
            out = self.demod.receive_batch(rx, llr_stride=648)
            self.last_n_llr, self.last_sync = out[1], out[2]
            return out[0]
        if self.kind == "dpsk":
            return self.demod.demod_soft_batch(rx, self.data_start, 1, llr_stride=648, llr=llr)
        if self.kind == "mcdpsk" and self.layout == "chirp":
            out = self.demod.chirp_receive_batch(rx, llr_stride=648)
            self.last_n_llr, self.last_sync, self.last_cfo = out[1], out[2], out[4]
            return out[0]
        return self.demod.demod_soft_batch(rx, llr_stride=648, llr=llr, want_cfo=False)[0]

    def _acquiring(self):
        return self.layout in ("sc", "chirp") or (self.kind == "dpsk" and self.acquire)

    def count_raw(self, llr, coded, index, bins, raw):
        """Raw counts of the first 648 soft bits of every row (decoder order); an acquiring receiver's n_llr marks the soft bits it did not
        deliver as erasures."""
        count_raw(self.ctx, llr, coded, raw, 648, self.last_n_llr if self._acquiring() else None, index, bins,
                  0 if self.kind == "ofdm" and self.layout == "presynced" else self.interleave_bps)

    def noise_std_table(self, snr_points):
        key = tuple(float(s) for s in snr_points)
        cache = self.__dict__.setdefault("_std_cache", {})
        if key not in cache:
            cache[key] = np.array([[channel_noise_std(self.tx_host[i], s, self.snr_convention) for i in range(self.pool)]
                                   for s in key], dtype=np.float32)
        return cache[key]

    @staticmethod
    def frame_seed(snr_idx, trial, base_seed=0xB200):
        return (np.uint64(base_seed) << np.uint64(40)) ^ (np.uint64(snr_idx) << np.uint64(32)) ^ np.uint64(trial)

    def make_batch(self, snr_points, snr_idx, trials, base_seed=0xB200):
        """Device descriptors of the frames (snr_idx[i], trials[i]): tx index, noise std, seed, counter bin."""
        import torch
        snr_idx = np.asarray(snr_idx, dtype=np.int64)
        trials = np.asarray(trials, dtype=np.int64)
        tx_index = (trials % self.pool).astype(np.uint32)
        std = self.noise_std_table(snr_points)[snr_idx, tx_index].astype(np.float32)
        seeds = ((np.uint64(base_seed) << np.uint64(40)) ^ (snr_idx.astype(np.uint64) << np.uint64(32))
                 ^ trials.astype(np.uint64))
        to = lambda a, dt: torch.from_numpy(a.view(dt) if a.dtype != dt else a).to(self.device)
        return dict(tx_index=to(tx_index.view(np.int32), np.int32), noise_std=to(std, np.float32),
                    seed=to(seeds.view(np.int64), np.int64), bins=to(snr_idx.astype(np.uint32).view(np.int32), np.int32),
                    host=dict(tx_index=tx_index, noise_std=std, seed=seeds, snr_idx=snr_idx))

    def fresh_frames(self, batch, snr_points):
        """Payloads drawn on the device (torch Philox stream keyed by the batch's first frame seed), pu_*_tx_batch, and the per-frame
        noise level of the tools' SNR convention.  Rows are built in the pool's order: chirp pair + body, peak normalisation over both,
        tools_cfo_hz through capi.ToolsCfo.  Returns (payload [B, kb] uint8 zero-padded, tx [B, L], noise_std [B])."""
        import torch
        B = batch["seed"].shape[0]
        g = torch.Generator(device=self.device)
        g.manual_seed(int(batch["host"]["seed"][0]) & 0x7FFFFFFFFFFFFFFF)
        kb = self.ldpc.info_bytes
        payload = torch.zeros((B, kb), dtype=torch.uint8, device=self.device)
        payload[:, :self.payload_bytes] = torch.randint(0, 256, (B, self.payload_bytes), dtype=torch.uint8, device=self.device, generator=g)
        # behind a chirp the peak is taken over chirp and body: the transmitter leaves the body unscaled
        peak = float(self.peak) if self.peak and self.chirp is None else 0.0
        if self.kind == "ofdm":
            tx = self.demod.tx_batch(self.ldpc, payload[:, :self.payload_bytes], layout=1 if self.layout == "sc" else 0, peak=peak)
        else:     # pu_dpsk_tx_batch / pu_mcdpsk_tx_batch
            tx = self.demod.tx_batch(self.ldpc, payload[:, :self.payload_bytes], peak=peak)
        if self.chirp is not None:
            tx = torch.nn.functional.pad(torch.cat([self.chirp.expand(B, -1), tx], dim=1), (self.lead, self.tail))
            if self.peak:
                tx = tx * (torch.tensor(float(self.peak), dtype=torch.float32, device=self.device) / tx.abs().amax(dim=1, keepdim=True))
        if self.tools_cfo_hz != 0.0:
            if self.tools_cfo is None or self.tools_cfo.n != tx.shape[1]:
                self.tools_cfo = capi.ToolsCfo(self.ctx, tx.shape[1], self.tools_cfo_hz, self.sample_rate)
            self.tools_cfo.apply_batch(tx)
        snr = np.asarray(snr_points, np.float32)
        fac = (np.power(np.float32(10.0), -snr / np.float32(20.0)) if self.snr_convention == 0
               else np.power(np.float32(10.0), snr / np.float32(10.0))).astype(np.float32)
        factor = torch.from_numpy(fac[batch["host"]["snr_idx"]]).to(self.device)
        std = torch.empty(B, dtype=torch.float32, device=self.device)
        capi.check(capi.lib().pu_channel_noise_std_batch(self.ctx._h, capi._ptr(tx), C.c_size_t(tx.stride(0)), C.c_size_t(tx.shape[1]),
                                                         C.c_size_t(B), capi._ptr(factor), int(self.snr_convention), capi._ptr(std),
                                                         C.c_void_p(torch.cuda.current_stream().cuda_stream)))
        return payload, tx, std

    def run_batch(self, batch, counters, rx=None, keep=False, snr_points=None, raw=None):
        """channel -> demod -> LDPC -> counters (and raw counts into `raw`) for one prepared batch (all on the current stream)."""
        if self.fresh_payload:
            import torch
            assert snr_points is not None, "fresh-payload batches need the SNR table to set each frame's noise level"
            payload, tx, std = self.fresh_frames(batch, snr_points)
            idx = torch.arange(tx.shape[0], dtype=torch.int32, device=self.device)
            rx = channel_apply(self.ctx, self.ch, tx, idx, std, batch["seed"], rx)
            coded = self.ldpc.encode_batch(payload[:, :self.payload_bytes]) if raw is not None else None
            if self.kind == "ofdm" and self.layout == "presynced" and raw is None:
                info, ok, iters = receive_decode(self.ofdm, self.ldpc, rx)
            elif self.kind == "ofdm" and self.layout == "presynced":
                llr = self.demod.presynced_batch(rx, 2, llr_stride=648, want_aux=False)[0]
                capi.count_raw_errors(self.ctx, llr, coded, raw, 648, None, None, batch["bins"], RAW_STRONG)
                info, ok, iters = self.ldpc.decode_batch(llr)
            else:
                llr = self.demod_llr(rx)
                if raw is not None:
                    self.count_raw(llr, coded, None, batch["bins"], raw)
                info, ok, iters = self.ldpc.decode_batch(llr)
                if self.layout in ("sc", "chirp") or (self.kind == "dpsk" and self.acquire):
                    ok = ok * (self.last_n_llr >= 648).to(ok.dtype)
            count_errors(self.ctx, info, ok, iters, payload, idx, batch["bins"], self.payload_bytes, counters)
            self.last_payload, self.last_tx, self.last_std = payload, tx, std
            return (rx, info, ok, iters) if keep else None
        rx = self.make_rx(batch, rx)
        info, ok, iters = self.receive_count(batch, rx, counters, raw=raw)
        return (rx, info, ok, iters) if keep else None

    def make_rx(self, batch, rx=None):
        """Channel outputs of a prepared batch (pool waveforms): pu_channel_apply_batch on the current stream."""
        return channel_apply(self.ctx, self.ch, self.tx_pool, batch["tx_index"], batch["noise_std"], batch["seed"], rx)

    def receive_count(self, batch, rx, counters, ev=None, bufs=None, raw=None):
        """demod -> LDPC -> counters for channel outputs `rx` of `batch`.  ev: optional list of >= 4 CUDA events recorded before the
        demodulator, between demodulator and decoder, behind the decoder and behind the counting kernel (bench.py's per-stage times).
        bufs: optional dict of preallocated device tensors {llr, info, ok, iters}.  raw: optional int64 [n_snr, 4] device tensor of
        RAW_COUNTER_NAMES, accumulated in place (the soft bits are counted between demodulator and decoder)."""
        bufs = bufs or {}
        rec = (lambda i: ev[i].record()) if ev is not None else (lambda i: None)
        count_raw = ((lambda llr: self.count_raw(llr, self.coded_pool, batch["tx_index"], batch["bins"], raw)) if raw is not None
                     else (lambda llr: None))
        rec(0)
        if self.kind == "ofdm" and self.layout in ("sc", "chirp"):
            # no sync or fewer than 648 soft bits is a lost frame (tools/test_mode_snr.cpp:72-77): the decoder's verdict on
            # the zero-filled row is overridden
            llr = self.demod_llr(rx)
            count_raw(llr)
            rec(1)
            info, ok, iters = self.ldpc.decode_batch(llr, bufs.get("info"), bufs.get("ok"), bufs.get("iters"))
            ok = ok * (self.last_n_llr >= 648).to(ok.dtype)
        elif self.kind == "ofdm" and ev is None and not bufs and raw is None:
            info, ok, iters = receive_decode(self.ofdm, self.ldpc, rx)
        elif self.kind == "ofdm":
            llr = bufs.get("llr")
            if llr is not None and self.ofdm.n_llr(rx.shape[1]) < 648:
                llr.zero_()                                              # frames shorter than a codeword: erasures
            llr = self.demod.presynced_batch(rx, 2, llr_stride=648, llr=llr, want_aux=False)[0]
            count_raw(llr)
            rec(1)
            info, ok, iters = self.ldpc.decode_batch(llr, bufs.get("info"), bufs.get("ok"), bufs.get("iters"))
        else:
            llr = self.demod_llr(rx, bufs.get("llr"))
            count_raw(llr)
            rec(1)
            info, ok, iters = self.ldpc.decode_batch(llr, bufs.get("info"), bufs.get("ok"), bufs.get("iters"))
            if (self.kind == "dpsk" and self.acquire) or (self.kind == "mcdpsk" and self.layout == "chirp"):
                ok = ok * (self.last_n_llr >= 648).to(ok.dtype)
        rec(2)
        count_errors(self.ctx, info, ok, iters, self.payload_pool, batch["tx_index"], batch["bins"], self.payload_bytes,
                     counters)
        rec(3)
        return info, ok, iters

    def sweep(self, snr_points, trials_per_point, rank=0, world=1, batch_frames=1 << 15, base_seed=0xB200, raw=False):
        """FER/BER sweep; this rank takes trials t with t % world == rank.  Returns an int64 [n_snr, 6] device tensor
        holding THIS rank's counters (all-reduce it with torch.distributed for the job total); raw=True returns (counters, raw [n_snr, 4])."""
        import torch
        counters = torch.zeros((len(snr_points), 6), dtype=torch.int64, device=self.device)
        table = torch.zeros((len(snr_points), 4), dtype=torch.int64, device=self.device) if raw else None
        mine = np.arange(rank, trials_per_point, world, dtype=np.int64)
        si = np.repeat(np.arange(len(snr_points), dtype=np.int64), len(mine))
        tr = np.tile(mine, len(snr_points))
        for off in range(0, len(si), batch_frames):
            b = self.make_batch(snr_points, si[off:off + batch_frames], tr[off:off + batch_frames], base_seed)
            self.run_batch(b, counters, snr_points=snr_points, raw=table)
        return (counters, table) if raw else counters


FRAME_COUNTER_NAMES = ("frames", "frame_errors", "codewords_failed", "codewords", "header_failures", "unused")
V2_BYTES_PER_CODEWORD = {capi.R1_4: 20, capi.R1_3: 27, capi.R1_2: 40, capi.R2_3: 54, capi.R3_4: 60, capi.R5_6: 67}


def v2_crc16(data):
    """CRC-16/CCITT (0x1021, init 0xFFFF) of src/protocol/frame_v2.cpp:111-124."""
    crc = 0xFFFF
    for b in bytes(data):
        crc ^= b << 8
        for _ in range(8):
            crc = ((crc << 1) ^ 0x1021) & 0xFFFF if crc & 0x8000 else (crc << 1) & 0xFFFF
    return crc


def v2_data_frame(payload, rate, seq=7, src_hash=0x123456, dst_hash=0xABCDEF, ftype=0x30, flags=0x01):
    """Bytes of a protocol-v2 DATA frame as DataFrame::serialize writes them (src/protocol/frame_v2.cpp:502-555): magic 0x554C, type,
    flags, seq, 24-bit source / destination hashes, TOTAL_CW (calculateCodewords, :439-460), payload length, header CRC, payload,
    frame CRC.  Only the simulator's stimulus: frame CONTENTS stay with the reference's protocol layer."""
    p = bytes(payload)
    total, bpc = 17 + len(p) + 2, V2_BYTES_PER_CODEWORD[rate]
    tcw = 1 if total <= bpc else 1 + -(-(total - bpc) // (bpc - 2))
    h = bytes([0x55, 0x4C, ftype, flags, seq >> 8, seq & 0xFF, src_hash >> 16, (src_hash >> 8) & 0xFF, src_hash & 0xFF,
               dst_hash >> 16, (dst_hash >> 8) & 0xFF, dst_hash & 0xFF, tcw, len(p) >> 8, len(p) & 0xFF])
    c = v2_crc16(h)
    body = h + bytes([c >> 8, c & 0xFF]) + p
    f = v2_crc16(body)
    return np.frombuffer(body + bytes([f >> 8, f & 0xFF]), np.uint8).copy()


class FrameLinkSim:
    """Whole-frame FER through the OFDM path (SURVEY §8f next-4 wired into the link simulation): every trial carries a protocol-v2 DATA
    frame of `payload_bytes` bytes = several LDPC codewords in one OFDM frame, and a trial succeeds iff RxPipeline::decodeFrame
    (src/gui/modem/rx_pipeline.cpp:348-445: CW0 -> header -> expected codewords -> all decoded -> reassemble) returns exactly the frame
    that was sent -- the reference's link-level statistic rather than the codeword FER of LinkSim.

        v2_data_frame -> pu_frame_encode -> pu_ofdm_tx (pool, host)  |  pu_channel_apply_batch -> pu_ofdm_presynced_batch (all
        codewords of the frame, llr_stride = n_cw * 648) -> pu_frame_decode_batch -> compare with the frame sent -> counters

    counters [n_snr, 6] = FRAME_COUNTER_NAMES.  payloads: explicit [pool, payload_bytes] array (e.g. the sweep driver's pool,
    capi.Sweep.payload; frame i then carries seq i + 1 as there); peak: the tools' peak normalisation of every TX waveform; interleave_bps > 0:
    ChannelInterleaver(interleave_bps, 648) on every codeword (interleave_codewords before modulating, capi.llr_deinterleave_batch on the
    soft bits of all codewords before decodeFrame), as the sweep driver's frame modes do.  raw: an int64 [n_snr, 4] device tensor given to
    run_batch accumulates RAW_COUNTER_NAMES over all n_cw * 648 soft bits of every frame (codewords the receiver did not deliver are
    erasures)."""

    def __init__(self, ctx, cfg, channel="awgn", payload_bytes=200, pool=16, pool_seed=12345, max_iter=50, precision="exact", code_rate=None,
                 payloads=None, peak=None, interleave_bps=0, layout="presynced", lead_samples=0, tail_samples=0):
        import torch
        assert isinstance(cfg, capi.ModemConfig), "whole frames ride on the OFDM waveforms"
        # layout "chirp": ChirpSync::generate() + training + data behind lead_samples of silence and ahead of tail_samples, received through
        # pu_ofdm_chirp_receive_batch; decodeFrame gets the whole codewords of soft bits the receiver delivered (the sweep driver's rule)
        assert layout in ("presynced", "chirp") and (layout == "chirp" or not (lead_samples or tail_samples))
        self.layout = layout
        self.ctx, self.cfg = ctx, cfg
        self.device = torch.device("cuda", ctx.device)
        self.ch = channel_preset(channel) if isinstance(channel, str) else channel
        self.snr_convention = 1 if channel == "awgn" else 0
        self.rate = cfg.code_rate if code_rate is None else code_rate
        self.ofdm = capi.OfdmDemodulator(ctx, cfg)
        self.ofdm.set_precision(precision)
        self.ldpc = capi.LdpcDecoder(ctx, self.rate, max_iter)
        if payloads is None:
            rng = np.random.default_rng(pool_seed)
            payloads = [rng.integers(0, 256, payload_bytes, dtype=np.uint8) for _ in range(pool)]
        else:
            payloads = np.ascontiguousarray(payloads, dtype=np.uint8).reshape(pool, payload_bytes)
        self.frames_host = [v2_data_frame(payloads[i], self.rate, seq=i + 1) for i in range(pool)]
        cws = [capi.frame_encode(self.rate, f) for f in self.frames_host]
        self.coded_pool = torch.from_numpy(np.stack([c.reshape(-1) for c in cws])).to(self.device)    # before interleaving: raw counts
        self.interleave_bps = int(interleave_bps)
        if self.interleave_bps:
            cws = [interleave_codewords(c, self.interleave_bps).reshape(c.shape) for c in cws]
        self.n_cw = len(cws[0])
        assert all(len(c) == self.n_cw for c in cws)
        waves = [ofdm_tx(cfg, c.reshape(-1), 0) for c in cws]
        if layout == "chirp":
            chirp = capi.chirp_generate(float(cfg.sample_rate), float(cfg.tx_cfo_hz))
            waves = [np.pad(np.concatenate([chirp, w]), (int(lead_samples), int(tail_samples))) for w in waves]
        if peak is not None:
            waves = [(w * (np.float32(peak) / np.abs(w).max())).astype(np.float32) for w in waves]
        self.tx_host = np.stack(waves)
        self.L = self.tx_host.shape[1]
        assert layout == "chirp" or self.ofdm.n_llr(self.L) >= self.n_cw * 648
        self.tx_pool = torch.from_numpy(self.tx_host).to(self.device)
        self.frame_len = len(self.frames_host[0])
        self.frame_pool = torch.from_numpy(np.stack(self.frames_host)).to(self.device)
        self.pool = pool

    def make_batch(self, snr_points, snr_idx, trials, base_seed=0xB200):
        import torch
        snr_idx = np.asarray(snr_idx, dtype=np.int64)
        trials = np.asarray(trials, dtype=np.int64)
        tx_index = (trials % self.pool).astype(np.uint32)
        table = np.array([[channel_noise_std(self.tx_host[i], s, self.snr_convention) for i in range(self.pool)] for s in snr_points], np.float32)
        std = table[snr_idx, tx_index].astype(np.float32)
        seeds = (np.uint64(base_seed) << np.uint64(40)) ^ (snr_idx.astype(np.uint64) << np.uint64(32)) ^ trials.astype(np.uint64)
        to = lambda a, dt: torch.from_numpy(a.view(dt) if a.dtype != dt else a).to(self.device)
        return dict(tx_index=to(tx_index.view(np.int32), np.int32), noise_std=to(std, np.float32), seed=to(seeds.view(np.int64), np.int64),
                    bins=to(snr_idx, np.int64), host=dict(tx_index=tx_index, noise_std=std, seed=seeds, snr_idx=snr_idx))

    def run_batch(self, batch, counters, keep=False, raw=None):
        """channel -> demod (every codeword of the frame) -> decodeFrame -> counters (and raw counts into `raw`), on the current stream."""
        import torch
        rx = channel_apply(self.ctx, self.ch, self.tx_pool, batch["tx_index"], batch["noise_std"], batch["seed"])
        if self.layout == "chirp":
            llr, n_llr = self.ofdm.chirp_receive_batch(rx, llr_stride=self.n_cw * 648)[:2]
        else:
            llr = self.ofdm.presynced_batch(rx, 2, llr_stride=self.n_cw * 648, want_aux=False)[0]
        if self.interleave_bps:
            capi.llr_deinterleave_batch(self.ctx, llr, self.n_cw, self.interleave_bps)
        if raw is not None:       # soft bits the chirp receiver did not deliver are erasures
            count_raw(self.ctx, llr, self.coded_pool, raw, self.n_cw * 648, n_llr if self.layout == "chirp" else None, batch["tx_index"],
                      batch["bins"].to(torch.int32), self.interleave_bps)
        frames, flen, info = self.ldpc.frame_decode_batch(llr, self.n_cw, frame_cap=self.frame_len)
        want = self.frame_pool[batch["tx_index"].long()]
        good = (info[:, 0] == 1) & (flen == self.frame_len) & (frames == want).all(dim=1)
        if self.layout == "chirp":
            # decodeFrame(soft_bits, num_codewords) with fewer codewords than the header expects: no codeword after CW0 is decoded and the
            # frame waits (rx_pipeline.cpp:394-401); without one whole codeword nothing is decoded at all (:352-354)
            short = n_llr < self.n_cw * 648
            none = n_llr < 648
            good = good & ~short
            info = info.clone()
            info[:, 3] = torch.where(short & (info[:, 2] > 0), 0, info[:, 3])
            info[:, 3] = torch.where(none, 0, info[:, 3])
            info[:, 4] = torch.where(none, 0, info[:, 4])
        upd = torch.stack([torch.ones_like(flen, dtype=torch.int64), (~good).to(torch.int64), info[:, 3].to(torch.int64),
                           torch.full_like(flen, self.n_cw, dtype=torch.int64), (info[:, 4] == 0).to(torch.int64),
                           torch.zeros_like(flen, dtype=torch.int64)], dim=1)
        counters.index_add_(0, batch["bins"], upd)
        return (rx, llr, frames, flen, info, good) if keep else None

    def sweep(self, snr_points, trials_per_point, rank=0, world=1, batch_frames=1 << 13, base_seed=0xB200, raw=False):
        import torch
        counters = torch.zeros((len(snr_points), 6), dtype=torch.int64, device=self.device)
        table = torch.zeros((len(snr_points), 4), dtype=torch.int64, device=self.device) if raw else None
        mine = np.arange(rank, trials_per_point, world, dtype=np.int64)
        si = np.repeat(np.arange(len(snr_points), dtype=np.int64), len(mine))
        tr = np.tile(mine, len(snr_points))
        for off in range(0, len(si), batch_frames):
            self.run_batch(self.make_batch(snr_points, si[off:off + batch_frames], tr[off:off + batch_frames], base_seed), counters, raw=table)
        return (counters, table) if raw else counters


def shard_trials(trials_per_point, rank, world):
    """Trial indices of this rank: t % world == rank (disjoint, exhaustive; no data-path collective, SURVEY §8e)."""
    return np.arange(rank, trials_per_point, world, dtype=np.int64)


def allreduce_counters(counters):
    """The path's only exchange step: sum the [n_snr, 6] int64 counter tables over all ranks (NCCL on GPUs, gloo in
    the CPU tests).  No-op without an initialised process group."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(counters, op=dist.ReduceOp.SUM)
    return counters


def summarize(counters, snr_points, raw=None):
    """Rows of {snr_db, frames, fer, ber, fer_ci, avg_iters} from a counter table (host).  With a raw table (RAW_COUNTER_NAMES) every row
    also has raw_ber = bit_errors / (soft_bits - erasures), erasure_rate = erasures / soft_bits and strong_error_share = strong_errors /
    bit_errors.  The raw BER has no confidence interval: the soft bits of one frame share its noise, fading and timing, so they are not
    independent trials and a binomial interval over bits would be far too narrow."""
    c = counters.detach().cpu().numpy() if hasattr(counters, "detach") else np.asarray(counters)
    r4 = None if raw is None else (raw.detach().cpu().numpy() if hasattr(raw, "detach") else np.asarray(raw))
    rows = []
    for i, (s, r) in enumerate(zip(snr_points, c)):
        frames, ferr, berr, bits, dfail, its = (int(v) for v in r)
        rows.append(dict(snr_db=float(s), frames=frames, fer=ferr / max(frames, 1), ber=berr / max(bits, 1),
                         fer_ci=wilson_interval(ferr, frames), decode_fail=dfail / max(frames, 1),
                         avg_iters=its / max(frames, 1)))
        if r4 is not None:
            soft, era, rerr, strong = (int(v) for v in r4[i])
            rows[-1].update(raw_ber=rerr / max(soft - era, 1), erasure_rate=era / max(soft, 1), strong_error_share=strong / max(rerr, 1))
    return rows
