"""Whole-frame FER in the sweep driver (pu_sweep_mode.frame_payload_bytes, csrc/sweep.cu) and its batched multi-codeword OFDM transmitter
(pu_frame_tx_batch, csrc/ofdm_tx_gpu.cu):
  - the transmitter is bit-identical to pu_frame_encode + pu_ofdm_tx, and equals pu_ofdm_tx_batch on one-codeword frames;
  - the driver's pool-path frame modes equal linksim.FrameLinkSim (pinned frame by frame to the oracle) counter for counter;
  - fresh frames agree with the pool within the binomial spread, are reproducible, shard over ranks and resume from a manifest;
  - a frame cannot beat a codeword, clean channels lose nothing, and an acquired frame short of soft bits is lost."""
import numpy as np
import pytest

import oracleapi as O
import refapi as R

pytestmark = pytest.mark.gpu

BPC = {R.R1_4: 20, R.R1_2: 40, R.R2_3: 54, R.R3_4: 60, R.R5_6: 67}


def words(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def frame_size(bpc, n):
    """Frame bytes that need n codewords with a partly filled last one."""
    return bpc - 5 if n == 1 else bpc + (n - 1) * (bpc - 2) - 3


@pytest.fixture(scope="module")
def ctx():
    from projectultra_b200 import capi
    c = capi.Context(0)
    yield c
    c.close()


PRESETS = {"m1_dqpsk": lambda r: R.config_m1(R.DQPSK, r), "m1_d8psk": lambda r: R.config_m1(R.D8PSK, r),
           "m1_16qam_p2": lambda r: R.config_m1(R.QAM16, r), "m3_32qam_p4": lambda r: R.config_m3(R.QAM32, r)}


@pytest.mark.parametrize("preset", sorted(PRESETS))
def test_frame_tx_batch_bit_identical(ctx, preset):
    import torch
    from projectultra_b200 import capi, linksim
    rng = np.random.default_rng(7)
    for rate, bpc in BPC.items():
        cfg = capi.ModemConfig.from_buffer_copy(bytes(PRESETS[preset](rate)))
        dem = capi.OfdmDemodulator(ctx, cfg)
        enc = capi.LdpcDecoder(ctx, rate)
        for n in (1, 2, 5, 41, 255):
            nbytes = frame_size(bpc, n)
            frames = rng.integers(0, 256, (2, nbytes), dtype=np.uint8)
            frames[1, : nbytes // 2] = 0
            for layout in (0, 1):
                coded = [capi.frame_encode(rate, f) for f in frames]
                assert all(len(c) == n for c in coded)
                want = np.stack([linksim.ofdm_tx(cfg, c.reshape(-1), layout) for c in coded])
                L = want.shape[1]
                # host memory, rows wider than a frame: the padding comes back as it went in
                out = np.full((2, L + 37), 3.5, np.float32)
                got, ncw = dem.frame_tx_batch(enc, frames, layout=layout, out=out)
                assert ncw == n
                assert (words(got[:, :L]) == words(want)).all(), (preset, rate, n, layout)
                assert (got[:, L:] == 3.5).all()
                # device memory, peak normalisation, padded rows
                dout = torch.full((2, L + 64), -1.0, dtype=torch.float32, device="cuda")
                dem.frame_tx_batch(enc, torch.from_numpy(frames).cuda(), layout=layout, peak=0.5, out=dout)
                torch.cuda.synchronize()
                scaled = np.stack([(w * (np.float32(0.5) / np.abs(w).max())).astype(np.float32) for w in want])
                d = dout.cpu().numpy()
                assert (words(d[:, :L]) == words(scaled)).all(), (preset, rate, n, layout, "peak")
                assert (d[:, L:] == -1.0).all()
                if n == 1:                     # the one-codeword case is pu_ofdm_tx_batch on the same bytes
                    one = dem.tx_batch(enc, frames, layout=layout)
                    assert (words(one) == words(want)).all()
                if n == 2 and layout == 1 and rate == R.R1_2:
                    assert (words(want[0]) == words(O.ofdm_tx(PRESETS[preset](rate), coded[0].reshape(-1), 1))).all()


def frame_counters(ctx, sw, mi, trials):
    """The same (mode, SNR point, trial) grid through linksim.FrameLinkSim with the driver's pool and seeds."""
    import torch
    from projectultra_b200 import capi, linksim
    m = sw.modes[mi]
    pool = sw.desc.pool
    payloads = np.stack([sw.payload(mi, i) for i in range(pool)])
    chan = [k for k, v in capi.CHANNELS.items() if v == m.channel][0]
    sim = linksim.FrameLinkSim(ctx, m.ofdm, chan, payload_bytes=m.frame_payload_bytes, pool=pool, code_rate=m.code_rate,
                               precision="fast" if m.precision else "exact", payloads=payloads, peak=m.peak or None)
    snrs = m.snr_points
    si = np.repeat(np.arange(len(snrs), dtype=np.int64), trials)
    tr = np.tile(np.arange(trials, dtype=np.int64), len(snrs))
    c = torch.zeros((len(snrs), 6), dtype=torch.int64, device="cuda")
    sim.run_batch(sim.make_batch(snrs, si, tr, base_seed=0xB200 | (mi << 16)), c)      # (mode << 56) of the driver's seed rule
    torch.cuda.synchronize()
    return c.cpu().numpy().astype(np.uint64), sim


def test_driver_frame_modes_match_frame_linksim(ctx):
    from projectultra_b200 import capi
    m1 = capi.ModemConfig.from_buffer_copy(bytes(R.config_m1(R.DQPSK, R.R1_2)))
    q16 = capi.ModemConfig.from_buffer_copy(bytes(R.config_m1(R.QAM16, R.R1_2)))
    modes = [capi.sweep_mode(capi.WF_OFDM, m1, R.R1_2, 0, "awgn", -2, 1.5, 4, frame_payload_bytes=60),                   # 3 CW, 35 symbols
             capi.sweep_mode(capi.WF_OFDM, m1, R.R1_2, 0, "awgn", -2, 1.5, 4, precision="fast", frame_payload_bytes=60),
             capi.sweep_mode(capi.WF_OFDM, q16, R.R1_2, 0, "good", 6, 3, 4, frame_payload_bytes=200),                      # 6 CW, pilots
             capi.sweep_mode(capi.WF_OFDM, q16, R.R1_2, 0, "good", 6, 3, 4, precision="fast", peak=0.5, frame_payload_bytes=200)]
    trials = 64
    sw = capi.Sweep(modes, trials_per_point=trials, block_trials=32, pool=8)
    counters, st = sw.run(ctx)
    assert st.units_run == sw.n_units and st.frames_run == trials * sw.n_points
    at = 0
    for mi, m in enumerate(modes):
        want, sim = frame_counters(ctx, sw, mi, trials)
        got = counters[at:at + m.n_snr]
        assert (got == want).all(), (mi, got.tolist(), want.tolist())
        assert (got[:, 0] == trials).all() and (got[:, 3] == trials * sim.n_cw).all() and (got[:, 5] == 0).all()
        # the short frames take the 512-FFT differential kernels (<= 40 symbols), the pilot mode the general presynced kernel
        short = ("ofdm_diff512_kernel", "ofdm_fast512_kernel")
        general = ("ofdm_presynced_kernel", "ofdm_presynced_warp_kernel", "ofdm_presynced_warp_fast_kernel")
        assert sim.ofdm.last_kernel in (short if mi < 2 else general), (mi, sim.ofdm.last_kernel)
        at += m.n_snr
    assert counters[0, 1] > counters[3, 1]                                      # a waterfall


def fresh_table(capi, fresh, snr_shift=0.0, chirp_channel="good"):
    m1 = capi.ModemConfig.from_buffer_copy(bytes(R.config_m1(R.DQPSK, R.R1_2)))
    kw = dict(peak=0.5, lead_samples=480, tail_samples=2400, fresh_payloads=fresh)
    return [capi.sweep_mode(capi.WF_OFDM, m1, R.R1_2, 0, "awgn", -1 + snr_shift, 1, 3, precision="fast", frame_payload_bytes=200, fresh_payloads=fresh),
            capi.sweep_mode(capi.WF_OFDM_SC, m1, R.R1_2, 0, "awgn", 8 + snr_shift, 2, 3, precision="fast", frame_payload_bytes=100, **kw),
            capi.sweep_mode(capi.WF_OFDM_CHIRP, m1, R.R1_2, 0, chirp_channel, 2 + snr_shift, 3, 3, precision="fast", frame_payload_bytes=100, **kw),
            capi.sweep_mode(capi.WF_OFDM_CHIRP, m1, R.R1_2, 0, "awgn", 1 + snr_shift, 2, 3, precision="fast", frame_payload_bytes=100, cfo_hz=30.0, **kw)]


def test_fresh_frames_match_the_pool_statistically(ctx, tmp_path):
    from projectultra_b200 import capi
    trials = 384
    kw = dict(trials_per_point=trials, block_trials=128, pool=32)
    pool, _ = capi.Sweep(fresh_table(capi, False), **kw).run(ctx)
    fresh, _ = capi.Sweep(fresh_table(capi, True), **kw).run(ctx)
    again, _ = capi.Sweep(fresh_table(capi, True), **kw).run(ctx)
    assert (fresh == again).all()
    parts = [capi.Sweep(fresh_table(capi, True), rank=r, world=2, **kw).run(ctx)[0] for r in range(2)]
    assert (parts[0] + parts[1] == fresh).all()
    assert (fresh[:, 0] == trials).all() and (fresh[:, 3] == pool[:, 3]).all()       # frames, codewords sent
    fp, ff = pool[:, 1] / trials, fresh[:, 1] / trials
    print("frame FER pool :", fp.round(3).tolist())
    print("frame FER fresh:", ff.round(3).tolist())
    sigma = np.sqrt(np.maximum(fp * (1 - fp), 0.02) * 2 / trials)
    assert (np.abs(fp - ff) < 5 * sigma + 0.02).all(), (fp - ff).tolist()
    # an interrupted fresh frame sweep resumes from its manifest to the uninterrupted totals
    d = str(tmp_path / "manifest")
    _, s1 = capi.Sweep(fresh_table(capi, True), manifest_dir=d, max_units=5, run_id=1, **kw).run(ctx)
    assert s1.units_run == 5
    tot = np.zeros_like(fresh)
    for r in range(2):
        c, st = capi.Sweep(fresh_table(capi, True), manifest_dir=d, rank=r, world=2, run_id=2, **kw).run(ctx)
        assert st.units_resumed == 5
        tot += c
    assert (tot == fresh).all()


def test_clean_frames_decode_and_a_frame_cannot_beat_a_codeword(ctx):
    from projectultra_b200 import capi
    clean, _ = capi.Sweep(fresh_table(capi, True, snr_shift=25.0, chirp_channel="awgn"), trials_per_point=128, block_trials=128, pool=8).run(ctx)
    assert (clean[:, 1] == 0).all() and (clean[:, 2] == 0).all() and (clean[:, 4] == 0).all(), clean.tolist()
    n_cw = {200: 6, 100: 4}                                                      # R1/2: 40 bytes in CW0, 38 in the others
    at = 0
    for m in fresh_table(capi, True):
        assert (clean[at:at + m.n_snr, 3] == 128 * n_cw[m.frame_payload_bytes]).all()
        at += m.n_snr
    # the bottom of the grid: frames of 6 codewords are lost at least as often as single codewords of the same modem and SNR
    m1 = capi.ModemConfig.from_buffer_copy(bytes(R.config_m1(R.DQPSK, R.R1_2)))
    q16 = capi.ModemConfig.from_buffer_copy(bytes(R.config_m1(R.QAM16, R.R1_2)))
    modes = [capi.sweep_mode(capi.WF_OFDM, m1, R.R1_2, 40, "awgn", -3, 1, 4, precision="fast"),
             capi.sweep_mode(capi.WF_OFDM, m1, R.R1_2, 0, "awgn", -3, 1, 4, precision="fast", frame_payload_bytes=200),
             capi.sweep_mode(capi.WF_OFDM, q16, R.R1_2, 40, "good", 6, 3, 4),
             capi.sweep_mode(capi.WF_OFDM, q16, R.R1_2, 0, "good", 6, 3, 4, frame_payload_bytes=200)]
    trials = 512
    c, _ = capi.Sweep(modes, trials_per_point=trials, block_trials=256, pool=32).run(ctx)
    fer = c[:, 1] / trials
    cw, fr = np.concatenate([fer[0:4], fer[8:12]]), np.concatenate([fer[4:8], fer[12:16]])
    print("codeword FER:", cw.round(3).tolist(), " frame FER:", fr.round(3).tolist())
    assert fr[0] > 0
    sigma = np.sqrt(np.maximum(cw * (1 - cw), 0.01) * 2 / trials)
    assert (fr > cw - 3 * sigma).all(), (fr - cw).tolist()


def test_acquired_frame_short_of_soft_bits_is_lost(ctx):
    """Without tail silence the delayed path of a Watterson channel pushes the last OFDM symbol out of the buffer: the chirp receiver
    returns fewer than n_cw * 648 soft bits, decodeFrame gets one codeword too few and waits -- the frame is lost, never "decoded" from
    a zero-filled codeword."""
    from projectultra_b200 import capi
    m1 = capi.ModemConfig.from_buffer_copy(bytes(R.config_m1(R.DQPSK, R.R1_4)))
    fer = {}
    for tail in (0, 2400):
        modes = [capi.sweep_mode(capi.WF_OFDM_CHIRP, m1, R.R1_4, 0, "good", 25, 5, 2, peak=0.5, precision="fast", lead_samples=480 if tail else 0,
                                 tail_samples=tail, frame_payload_bytes=100, fresh_payloads=True)]
        c, _ = capi.Sweep(modes, trials_per_point=128, block_trials=128, pool=8).run(ctx)
        fer[tail] = c[:, 1] / c[:, 0]
    print("frame FER without / with tail silence:", fer[0].tolist(), fer[2400].tolist())
    assert (fer[0] > 0.7).all() and (fer[2400] < 0.1).all()
