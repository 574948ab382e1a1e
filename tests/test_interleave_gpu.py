"""ChannelInterleaver(bps, 648) on every codeword (the reference's IWaveform path: getSoftBits -> ChannelInterleaver::deinterleave ->
decodeSoft), on the GPU:
  - pu_llr_deinterleave_batch equals the oracle's deinterleave block by block, in device and host memory, and leaves padding alone;
  - the transmitters with pu_*_set_tx_interleave equal encode -> byte interleave -> host modulator, and reproduce their old output at 0;
  - the sweep driver with pu_sweep_mode.interleave_bps equals linksim.LinkSim / FrameLinkSim counter for counter on Watterson channels;
  - fresh frames agree with the pool, and both halves of the interleaver are needed to decode."""
import numpy as np
import pytest

import oracleapi as O
import refapi as R

pytestmark = pytest.mark.gpu

BPC = {R.R1_4: 20, R.R1_2: 40, R.R2_3: 54, R.R3_4: 60, R.R5_6: 67}
PRESETS = {"m1_dqpsk": lambda r: R.config_m1(R.DQPSK, r), "m1_d8psk": lambda r: R.config_m1(R.D8PSK, r),
           "m1_16qam_p2": lambda r: R.config_m1(R.QAM16, r), "m3_32qam_p4": lambda r: R.config_m3(R.QAM32, r)}


def words(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def interleave_bytes(coded, bps):
    """ChannelInterleaver::interleave of every 81-byte codeword: bit i of a codeword goes to bit perm[i] (MSB first)."""
    from projectultra_b200 import capi
    perm = capi.channel_interleaver_perm(bps)[0]
    bits = np.unpackbits(np.asarray(coded, np.uint8).reshape(-1, 81), axis=1)
    out = np.zeros_like(bits)
    out[:, perm] = bits
    return np.packbits(out, axis=1).reshape(-1)


@pytest.fixture(scope="module")
def ctx():
    from projectultra_b200 import capi
    c = capi.Context(0)
    yield c
    c.close()


@pytest.mark.parametrize("bps", [1, 16, 40, 60, 90, 118, 220, 512])
def test_llr_deinterleave_matches_the_oracle(ctx, bps):
    import torch
    from projectultra_b200 import capi
    rng = np.random.default_rng(bps)
    for n_blocks, B in ((1, 37), (2, 5), (7, 3), (255, 3)):
        stride = n_blocks * 648 + 11                           # padding behind the blocks must not be written
        x = rng.standard_normal((B, stride)).astype(np.float32)
        if n_blocks > 1:
            x[1, 648:2 * 648] = 0.0                            # an erasure block stays an erasure
        want = x.copy()
        for b in range(B):
            for c in range(n_blocks):
                want[b, c * 648:(c + 1) * 648] = O.channel_interleave(bps, x[b, c * 648:(c + 1) * 648], inverse=True)
        host = capi.llr_deinterleave_batch(ctx, x.copy(), n_blocks, bps)
        assert (words(host) == words(want)).all(), (bps, n_blocks, "host")
        dev = capi.llr_deinterleave_batch(ctx, torch.from_numpy(x).cuda(), n_blocks, bps)
        torch.cuda.synchronize()
        assert (words(dev.cpu().numpy()) == words(want)).all(), (bps, n_blocks, "device")
        if n_blocks > 1:
            assert (host[1, 648:2 * 648] == 0).all()
        # interleave (oracle) then deinterleave (GPU) is the identity
        inter = x.copy()
        for b in range(B):
            for c in range(n_blocks):
                inter[b, c * 648:(c + 1) * 648] = O.channel_interleave(bps, x[b, c * 648:(c + 1) * 648])
        assert (words(capi.llr_deinterleave_batch(ctx, inter, n_blocks, bps)) == words(x)).all()


def test_llr_deinterleave_rejects_blocks_beyond_the_row(ctx):
    from projectultra_b200 import capi
    with pytest.raises(capi.PuError):
        capi.llr_deinterleave_batch(ctx, np.zeros((2, 1000), np.float32), 2, 60)
    with pytest.raises(capi.PuError):
        capi.llr_deinterleave_batch(ctx, np.zeros((2, 648), np.float32), 1, 0)


@pytest.mark.parametrize("preset", sorted(PRESETS))
def test_ofdm_transmitters_interleave_every_codeword(ctx, preset):
    import torch
    from projectultra_b200 import capi, linksim
    rng = np.random.default_rng(11)
    for rate, bpc in BPC.items():
        cfg = capi.ModemConfig.from_buffer_copy(bytes(PRESETS[preset](rate)))
        dem = capi.OfdmDemodulator(ctx, cfg)
        enc = capi.LdpcDecoder(ctx, rate)
        bps = dem.bits_per_symbol
        for n in (1, 2, 7, 255):
            nbytes = bpc - 5 if n == 1 else bpc + (n - 1) * (bpc - 2) - 3
            frames = rng.integers(0, 256, (2, nbytes), dtype=np.uint8)
            coded = [capi.frame_encode(rate, f) for f in frames]
            for layout in (0, 1):
                want = np.stack([linksim.ofdm_tx(cfg, interleave_bytes(c, bps), layout) for c in coded])
                plain = np.stack([linksim.ofdm_tx(cfg, c.reshape(-1), layout) for c in coded])
                L = want.shape[1]
                dem.set_tx_interleave(bps)
                got, ncw = dem.frame_tx_batch(enc, frames, layout=layout)
                assert ncw == n and (words(got) == words(want)).all(), (preset, rate, n, layout)
                dout = torch.full((2, L + 64), -1.0, dtype=torch.float32, device="cuda")
                dem.frame_tx_batch(enc, torch.from_numpy(frames).cuda(), layout=layout, peak=0.5, out=dout)
                torch.cuda.synchronize()
                scaled = np.stack([(w * (np.float32(0.5) / np.abs(w).max())).astype(np.float32) for w in want])
                d = dout.cpu().numpy()
                assert (words(d[:, :L]) == words(scaled)).all() and (d[:, L:] == -1.0).all(), (preset, rate, n, layout, "peak")
                if n == 1:
                    assert (words(dem.tx_batch(enc, frames, layout=layout)) == words(want)).all()
                dem.set_tx_interleave(0)
                assert (words(dem.frame_tx_batch(enc, frames, layout=layout)[0]) == words(plain)).all()
                if n == 1:
                    assert (words(dem.tx_batch(enc, frames, layout=layout)) == words(plain)).all()


@pytest.mark.parametrize("nc", [3, 8, 20])
@pytest.mark.parametrize("bits", [1, 2])
def test_mcdpsk_transmitter_interleaves_the_codeword(ctx, nc, bits):
    import torch
    from projectultra_b200 import capi
    rng = np.random.default_rng(nc * 10 + bits)
    cfg = capi.mcdpsk_config(nc, bits)
    dem = capi.McDpskDemodulator(ctx, cfg)
    enc = capi.LdpcDecoder(ctx, capi.R1_2)
    payload = rng.integers(0, 256, (4, 40), dtype=np.uint8)
    coded = [capi.ldpc_encode(capi.R1_2, p) for p in payload]
    want = np.stack([capi.mcdpsk_tx(cfg, interleave_bytes(c, nc * bits)) for c in coded])
    plain = np.stack([capi.mcdpsk_tx(cfg, c) for c in coded])
    dem.set_tx_interleave(nc * bits)
    assert (words(dem.tx_batch(enc, payload)) == words(want)).all()
    d = dem.tx_batch(enc, torch.from_numpy(payload).cuda(), peak=0.5)
    torch.cuda.synchronize()
    scaled = np.stack([(w * (np.float32(0.5) / np.abs(w).max())).astype(np.float32) for w in want])
    assert (words(d.cpu().numpy()) == words(scaled)).all()
    dem.set_tx_interleave(0)
    assert (words(dem.tx_batch(enc, payload)) == words(plain)).all()


def cfg_m1(capi, rate=R.R1_2):
    return capi.ModemConfig.from_buffer_copy(bytes(R.config_m1(R.DQPSK, rate)))


SILENCE = dict(peak=0.5, lead_samples=480, tail_samples=2400)


def codeword_table(capi):
    mc = capi.mcdpsk_config(8, 2)
    return [capi.sweep_mode(capi.WF_OFDM, cfg_m1(capi), R.R1_2, 40, "moderate", 2, 3, 4, interleave_bps=60),
            capi.sweep_mode(capi.WF_OFDM, cfg_m1(capi), R.R1_2, 40, "moderate", 2, 3, 4, precision="fast", interleave_bps=60),
            capi.sweep_mode(capi.WF_OFDM_CHIRP, cfg_m1(capi), R.R1_2, 40, "good", 2, 3, 4, precision="fast", interleave_bps=60, **SILENCE),
            capi.sweep_mode(capi.WF_MCDPSK, mc, R.R1_2, 40, "moderate", 0, 3, 4, peak=0.5, interleave_bps=16),
            capi.sweep_mode(capi.WF_MCDPSK_CHIRP, mc, R.R1_2, 40, "moderate", 0, 3, 4, interleave_bps=16, **SILENCE)]


def linksim_counters(ctx, sw, mi, trials):
    import torch
    from projectultra_b200 import capi, linksim
    m = sw.modes[mi]
    pool = sw.desc.pool
    payloads = np.stack([sw.payload(mi, i) for i in range(pool)])
    cfg = m.ofdm if m.waveform <= capi.WF_OFDM_CHIRP else m.mcdpsk
    chan = [k for k, v in capi.CHANNELS.items() if v == m.channel][0]
    chirp = m.waveform in (capi.WF_OFDM_CHIRP, capi.WF_MCDPSK_CHIRP)
    sim = linksim.LinkSim(ctx, cfg, chan, payload_bytes=m.payload_bytes, pool=pool, code_rate=m.code_rate, peak=m.peak or None,
                          precision="fast" if m.precision else "exact", payloads=payloads, layout="chirp" if chirp else "presynced",
                          lead_samples=m.lead_samples, tail_samples=m.tail_samples, interleave_bps=m.interleave_bps)
    snrs = m.snr_points
    si = np.repeat(np.arange(len(snrs), dtype=np.int64), trials)
    tr = np.tile(np.arange(trials, dtype=np.int64), len(snrs))
    c = torch.zeros((len(snrs), 6), dtype=torch.int64, device="cuda")
    sim.run_batch(sim.make_batch(snrs, si, tr, base_seed=0xB200 | (mi << 16)), c)      # (mode << 56) of the driver's seed rule
    torch.cuda.synchronize()
    return c.cpu().numpy().astype(np.uint64), sim


def test_driver_matches_linksim_with_interleaving(ctx):
    from projectultra_b200 import capi
    trials = 96
    modes = codeword_table(capi)
    sw = capi.Sweep(modes, trials_per_point=trials, block_trials=48, pool=8)
    counters, _ = sw.run(ctx)
    at = 0
    for mi, m in enumerate(modes):
        want, sim = linksim_counters(ctx, sw, mi, trials)
        got = counters[at:at + m.n_snr]
        assert (got == want).all(), (mi, got.tolist(), want.tolist())
        assert (got[:, 0] == trials).all()
        if mi < 2:       # PU_WF_OFDM codewords take the fused table of the 512-FFT differential kernels
            assert sim.ofdm.last_kernel == ("ofdm_diff512_kernel" if mi == 0 else "ofdm_fast512_kernel")
        at += m.n_snr
    print("FER interleaved:", (counters[:, 1] / trials).round(3).tolist())
    assert counters[0, 1] > counters[3, 1]                                       # a waterfall on the moderate channel
    # on a fading channel the interleaver changes which frames fail
    modes[0].interleave_bps = 0
    off, _ = capi.Sweep(modes[:1], trials_per_point=trials, block_trials=48, pool=8).run(ctx)
    assert not (off == counters[:4]).all()


def frame_table(capi):
    q16 = capi.ModemConfig.from_buffer_copy(bytes(R.config_m1(R.QAM16, R.R1_2)))
    return [capi.sweep_mode(capi.WF_OFDM, cfg_m1(capi), R.R1_2, 0, "good", 0, 3, 4, precision="fast", frame_payload_bytes=60, interleave_bps=60),
            capi.sweep_mode(capi.WF_OFDM, q16, R.R1_2, 0, "good", 6, 3, 4, frame_payload_bytes=200, interleave_bps=112),
            capi.sweep_mode(capi.WF_OFDM_CHIRP, cfg_m1(capi), R.R1_2, 0, "moderate", 2, 3, 4, precision="fast", frame_payload_bytes=100,
                            interleave_bps=60, **SILENCE)]


def test_driver_frame_modes_match_frame_linksim_with_interleaving(ctx):
    import torch
    from projectultra_b200 import capi, linksim
    trials = 64
    modes = frame_table(capi)
    sw = capi.Sweep(modes, trials_per_point=trials, block_trials=32, pool=8)
    counters, _ = sw.run(ctx)
    at = 0
    for mi, m in enumerate(modes):
        payloads = np.stack([sw.payload(mi, i) for i in range(8)])
        chan = [k for k, v in capi.CHANNELS.items() if v == m.channel][0]
        chirp = m.waveform == capi.WF_OFDM_CHIRP
        sim = linksim.FrameLinkSim(ctx, m.ofdm, chan, payload_bytes=m.frame_payload_bytes, pool=8, code_rate=m.code_rate,
                                   precision="fast" if m.precision else "exact", payloads=payloads, peak=m.peak or None,
                                   interleave_bps=m.interleave_bps, layout="chirp" if chirp else "presynced", lead_samples=m.lead_samples,
                                   tail_samples=m.tail_samples)
        snrs = m.snr_points
        si = np.repeat(np.arange(len(snrs), dtype=np.int64), trials)
        tr = np.tile(np.arange(trials, dtype=np.int64), len(snrs))
        c = torch.zeros((len(snrs), 6), dtype=torch.int64, device="cuda")
        sim.run_batch(sim.make_batch(snrs, si, tr, base_seed=0xB200 | (mi << 16)), c)
        torch.cuda.synchronize()
        want = c.cpu().numpy().astype(np.uint64)
        got = counters[at:at + m.n_snr]
        assert (got == want).all(), (mi, got.tolist(), want.tolist())
        assert (got[:, 0] == trials).all() and (got[:, 3] == trials * sim.n_cw).all()
        at += m.n_snr
    print("frame FER interleaved:", (counters[:, 1] / trials).round(3).tolist())
    assert counters[0, 1] > counters[3, 1]


def test_fresh_interleaved_frames_match_the_pool(ctx):
    from projectultra_b200 import capi

    def table(fresh):
        t = codeword_table(capi)[1:] + frame_table(capi)[::2]
        for m in t:
            m.fresh_payloads = int(fresh)
        return t

    trials = 384
    kw = dict(trials_per_point=trials, block_trials=128, pool=32)
    pool, _ = capi.Sweep(table(False), **kw).run(ctx)
    fresh, _ = capi.Sweep(table(True), **kw).run(ctx)
    again, _ = capi.Sweep(table(True), **kw).run(ctx)
    assert (fresh == again).all()
    assert (fresh[:, 0] == trials).all() and (fresh[:, 3] == pool[:, 3]).all()
    fp, ff = pool[:, 1] / trials, fresh[:, 1] / trials
    print("FER pool :", fp.round(3).tolist())
    print("FER fresh:", ff.round(3).tolist())
    sigma = np.sqrt(np.maximum(fp * (1 - fp), 0.02) * 2 / trials)
    assert (np.abs(fp - ff) < 5 * sigma + 0.02).all(), (fp - ff).tolist()


def test_both_halves_of_the_interleaver_are_wired(ctx):
    import torch
    from projectultra_b200 import capi, linksim
    # clean high-SNR AWGN loses nothing with interleaving on, in every waveform and in frame mode
    modes = []
    for m in codeword_table(capi) + frame_table(capi):
        m.channel, m.snr_first_db, m.n_snr = capi.CHANNELS["awgn"], 25.0, 1
        modes.append(m)
    for fresh in (False, True):
        for m in modes:
            m.fresh_payloads = int(fresh)
        c, _ = capi.Sweep(modes, trials_per_point=128, block_trials=128, pool=8).run(ctx)
        assert (c[:, 0] == 128).all() and (c[:, 1] == 0).all(), (fresh, c.tolist())
    # an interleaved pool waveform decodes through the deinterleaver and fails without it
    cfg = cfg_m1(capi)
    sim = linksim.LinkSim(ctx, cfg, "awgn", payload_bytes=40, pool=16, code_rate=R.R1_2, interleave_bps=60)
    rx = sim.tx_pool.clone()
    info, ok, _ = linksim.receive_decode(sim.ofdm, sim.ldpc, rx)
    assert bool(ok.all()) and (info[:, :40].cpu().numpy() == sim.payloads).all()
    sim.ofdm.set_deinterleave(0)
    info, ok, _ = linksim.receive_decode(sim.ofdm, sim.ldpc, rx)
    assert not bool(ok.any()) or not (info[:, :40].cpu().numpy() == sim.payloads).all(axis=1).any()
    llr = sim.ofdm.presynced_batch(rx, 2, llr_stride=648, want_aux=False)[0]
    info, ok, _ = sim.ldpc.decode_batch(capi.llr_deinterleave_batch(ctx, llr, 1, 60))
    assert bool(ok.all()) and (info[:, :40].cpu().numpy() == sim.payloads).all()
    torch.cuda.synchronize()
