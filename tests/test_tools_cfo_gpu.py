"""The tools' FFT-Hilbert CFO injector on the GPU (pu_tools_cfo_*, csrc/tools_cfo_gpu.cu) and the fresh-payload transmit chain it completes:
batched rows bit for bit against the host function (csrc/tools_cfo.cpp) and the plain-C oracle, the chirp-fronted fresh frames of LinkSim
bit for bit against the host transmitter, and the sweep driver's fresh payloads on the chirp-acquired and tuning-error modes."""
import numpy as np
import pytest

import channelapi as CH
import oracleapi as O
import refapi as R

pytestmark = pytest.mark.gpu

SENTINEL = np.uint32(0x7FC0BEEF)        # a NaN pattern in the padding between n and stride: any write shows


@pytest.fixture(scope="module")
def ctx():
    from projectultra_b200 import capi
    c = capi.Context(0)
    yield c
    c.close()


def rows(n, B, stride, seed):
    rng = np.random.default_rng(seed)
    x = np.full((B, stride), SENTINEL, np.uint32).view(np.float32)
    t = np.arange(n) / 48000.0
    for b in range(B):
        f = 700.0 + 90.0 * b
        x[b, :n] = (0.4 * np.sin(2 * np.pi * f * t + 0.3 * b) + 0.05 * rng.standard_normal(n)).astype(np.float32)
    x[0, :min(n, 300)] = 0.0                                   # silence in front, as the sweep's rows have
    return x


def batch_rows(n):
    """More rows than one pass of the two-pass schedule holds (64 MiB of scratch = 2^22 / P rows), a few for one-CTA rows."""
    P = 1 << max(0, (n - 1).bit_length())
    return (1 << 22) // P + 1 if P > 8192 else 3


@pytest.mark.parametrize("cfo", [30.0, -50.0, 12.5, 0.0005])
@pytest.mark.parametrize("n", [127, 128, 5000, 65536, 65537, 68812, 87080, 204200, 1 << 20])
def test_batch_matches_the_host_injector_bit_for_bit(ctx, n, cfo):
    import torch
    from projectultra_b200 import capi
    B, stride = batch_rows(n), n + 37
    x = rows(n, B, stride, n)
    want = np.stack([capi.tools_apply_cfo(x[b, :n], cfo) for b in range(B)])
    for b in (0, B - 1):
        assert (O.tools_apply_cfo(x[b, :n], cfo).view(np.uint32) == want[b].view(np.uint32)).all(), b
    h = capi.ToolsCfo(ctx, n, cfo)
    launches = ctx.kernel_launches
    dev = torch.from_numpy(x.copy()).cuda()
    h.apply_batch(dev)
    got_dev = dev.cpu().numpy()
    got_host = h.apply_batch(x.copy())
    noop = n < 128 or abs(cfo) < 0.001
    assert (ctx.kernel_launches == launches) == noop
    for got in (got_dev, got_host):
        assert (got[:, n:].view(np.uint32) == SENTINEL).all(), "padding between n and stride written"
        bad = np.nonzero((got[:, :n].view(np.uint32) != want.view(np.uint32)).any(axis=1))[0]
        assert len(bad) == 0, (bad.tolist(), np.abs(got[bad[0], :n] - want[bad[0]]).max())
        if noop:
            assert (got.view(np.uint32) == x.view(np.uint32)).all()
    h.close()


def test_limits_and_bad_arguments(ctx):
    import ctypes as C
    from projectultra_b200 import capi
    with pytest.raises(capi.PuError, match="unsupported"):
        capi.ToolsCfo(ctx, (1 << 20) + 1, 30.0)
    for bad in [(1000, 30.0, 0.0), (1000, float("nan"), 48000.0)]:
        with pytest.raises(capi.PuError, match="invalid"):
            capi.ToolsCfo(ctx, *bad)
    h = capi.ToolsCfo(ctx, 1000, 30.0)
    with pytest.raises(capi.PuError, match="invalid"):
        h.apply_batch(np.zeros((2, 999), np.float32))                          # stride shorter than a row
    L = capi.lib()
    assert L.pu_tools_cfo_apply_batch(h._h, None, C.c_size_t(2), C.c_size_t(1000), capi.PU_MEM_HOST, None) == 1
    assert L.pu_tools_cfo_apply_batch(h._h, None, C.c_size_t(0), C.c_size_t(1000), capi.PU_MEM_HOST, None) == 0
    assert L.pu_tools_cfo_apply_batch(None, None, C.c_size_t(0), C.c_size_t(1000), capi.PU_MEM_HOST, None) == 1
    x = np.ones((1, 1000), np.float32)
    assert L.pu_tools_cfo_apply_batch(h._h, capi._ptr(x), C.c_size_t(1), C.c_size_t(1000), 7, None) == 1
    out = C.c_void_p()
    assert L.pu_tools_cfo_create(None, C.c_size_t(1000), C.c_float(30.0), C.c_float(48000.0), C.byref(out)) == 1
    h.close()


@pytest.mark.parametrize("kind,cfo", [("ofdm", 30.0), ("ofdm", -30.0), ("mcdpsk", 30.0), ("mcdpsk", -30.0)])
def test_fresh_chirp_frames_are_the_host_transmit_chain(ctx, kind, cfo):
    """LinkSim(layout='chirp', fresh_payload=True, peak, tools_cfo_hz, silence): every row is silence + chirp + host TX(payload) + silence
    -> peak -> pu_tools_apply_cfo, bit for bit; the noise level follows the tools' convention; frames at high SNR decode."""
    import torch
    from projectultra_b200 import capi, linksim
    if kind == "ofdm":
        rcfg = R.config_m1(R.DQPSK, R.R1_2)
        cfg, rate, pb = capi.ModemConfig.from_buffer_copy(bytes(rcfg)), capi.R1_2, 40
        chirp = capi.chirp_generate(48000.0, float(cfg.tx_cfo_hz))
        body = lambda coded: linksim.ofdm_tx(cfg, coded, 0)
    else:
        cfg, rate, pb = capi.mcdpsk_config(8, 2), capi.R1_2, 40
        chirp = capi.chirp_generate(48000.0, 0.0)
        body = lambda coded: capi.mcdpsk_tx(cfg, coded)
    lead, tail = 480, 2400                  # the sweep's silence: a +30 Hz error moves the up chirp's apparent start in front of the frame
    sim = linksim.LinkSim(ctx, cfg, "awgn", payload_bytes=pb, pool=2, code_rate=rate, peak=0.5, layout="chirp", fresh_payload=True,
                          tools_cfo_hz=cfo, precision="fast" if kind == "ofdm" else "exact", lead_samples=lead, tail_samples=tail)
    snrs = [30.0]
    trials = 12
    batch = sim.make_batch(snrs, np.zeros(trials, np.int64), np.arange(trials))
    counters = torch.zeros((1, 6), dtype=torch.int64, device="cuda")
    sim.run_batch(batch, counters, snr_points=snrs)
    torch.cuda.synchronize()
    payload, tx, std = sim.last_payload.cpu().numpy(), sim.last_tx.cpu().numpy(), sim.last_std.cpu().numpy()
    assert len(np.unique(payload[:, :pb], axis=0)) == trials
    for b in range(trials):
        w = np.concatenate([np.zeros(lead, np.float32), chirp, body(capi.ldpc_encode(rate, payload[b, :pb])), np.zeros(tail, np.float32)])
        w = (w * (np.float32(0.5) / np.abs(w).max())).astype(np.float32)
        w = capi.tools_apply_cfo(w, cfo)
        assert (w.view(np.uint32) == tx[b].view(np.uint32)).all(), b
        assert abs(std[b] - CH.noise_std(w, snrs[0], 1)) <= 2e-7 * std[b], (b, std[b])
    c = counters.cpu().numpy()
    assert c[0, 0] == trials and c[0, 1] == 0, c.tolist()


def test_fresh_payloads_on_the_chirp_and_tuning_error_modes(ctx):
    """pu_sweep_mode.fresh_payloads on the chirp-acquired waveforms with the tools' tuning error (the regression matrix's --cfo rows):
    reproducible, two ranks sum to the single-rank table, the FER agrees with the pool's within the binomial spread, the matrix's rows
    decode, and a 30 Hz error in front of the genie-timed receiver (no chirp estimate) loses the frames -- the injector runs."""
    from projectultra_b200 import capi
    m1 = capi.ModemConfig.from_buffer_copy(bytes(R.config_m1(R.DQPSK, R.R1_2)))
    mc = capi.mcdpsk_config(8, 2)
    kw = dict(peak=0.5, lead_samples=480, tail_samples=2400)

    def table(fresh):
        t = [capi.sweep_mode(capi.WF_OFDM_CHIRP, m1, capi.R1_2, 40, "awgn", 5, 12, 2, precision="fast", cfo_hz=c, fresh_payloads=fresh, **kw)
             for c in (0.0, 30.0, -30.0)]
        t += [capi.sweep_mode(capi.WF_MCDPSK_CHIRP, mc, capi.R1_2, 40, "awgn", -3, 8, 2, cfo_hz=c, fresh_payloads=fresh, **kw) for c in (0.0, 30.0, -30.0)]
        t += [capi.sweep_mode(capi.WF_MCDPSK, mc, capi.R1_2, 40, "awgn", 5, 1, 1, cfo_hz=30.0, peak=0.5, fresh_payloads=fresh)]
        return t

    trials = 256
    run = lambda fresh, **a: capi.Sweep(table(fresh), trials_per_point=trials, block_trials=64, pool=16, **a).run(ctx)[0]
    pool, fresh, again = run(False), run(True), run(True)
    assert (fresh == again).all()
    parts = [run(True, rank=r, world=2) for r in range(2)]
    assert (parts[0] + parts[1] == fresh).all()
    assert (fresh[:, 0] == trials).all() and (fresh[:, 3] == pool[:, 3]).all()
    fp, ff = pool[:, 1] / trials, fresh[:, 1] / trials
    print("FER pool :", fp.round(3).tolist())
    print("FER fresh:", ff.round(3).tolist())
    sigma = np.sqrt(np.maximum(fp * (1 - fp), 0.02) * 2 / trials)
    assert (np.abs(fp - ff) < 5 * sigma + 0.02).all(), (fp - ff).tolist()
    matrix_rows = [1, 3, 5, 7, 9, 11]                 # OFDM_CHIRP at 17 dB, MC-DPSK behind the chirp at 5 dB, cfo 0 / 30 / -30
    assert (ff[matrix_rows] < 0.1).all(), ff.tolist()
    assert ff[12] > 0.9, ff.tolist()
