"""Pre-decoder (raw) bit error counts: the batched LDPC / frame encoder on the GPU (pu_ldpc_encode_batch, pu_frame_encode_batch), the raw
error counter (pu_count_raw_errors) and the sweep driver's raw table (pu_linksim_run_raw):
  - the encoders are bit-identical to the host encoders in device and host memory, with padded rows and the codeword-count query;
  - the counter equals a numpy count on rows with +-0, +-10, values either side of `strong`, short rows, bins and gathers;
  - the driver's raw table equals LinkSim / FrameLinkSim counter for counter on the pool path, and its 6-column table is unchanged;
  - fresh trials agree with the pool, are reproducible, shard over ranks, resume from a raw manifest and refuse a plain one;
  - raw BER is 1/2 far below the waterfall, 0 far above it, and an acquired frame short of soft bits shows its erasures."""
import os

import numpy as np
import pytest

import refapi as R

pytestmark = pytest.mark.gpu

RATES = (R.R1_4, R.R1_3, R.R1_2, R.R2_3, R.R3_4, R.R5_6, R.R7_8)
BPC = {R.R1_4: 20, R.R1_3: 27, R.R1_2: 40, R.R2_3: 54, R.R3_4: 60, R.R5_6: 67, R.R7_8: 20}


@pytest.fixture(scope="module")
def ctx():
    from projectultra_b200 import capi
    c = capi.Context(0)
    yield c
    c.close()


def frame_size(bpc, n):
    """Frame bytes that need n codewords with a partly filled last one."""
    return bpc - 5 if n == 1 else bpc + (n - 1) * (bpc - 2) - 3


@pytest.mark.parametrize("rate", RATES)
def test_ldpc_encode_batch_bit_identical(ctx, rate):
    import torch
    from projectultra_b200 import capi
    enc = capi.LdpcDecoder(ctx, rate)
    rng = np.random.default_rng(rate)
    for n in range(1, enc.k // 8 + 1):
        pay = rng.integers(0, 256, (3, n), dtype=np.uint8)
        want = np.stack([capi.ldpc_encode(rate, p) for p in pay])
        assert want.shape == (3, 81)
        got = enc.encode_batch(torch.from_numpy(pay).cuda())
        torch.cuda.synchronize()
        assert (got.cpu().numpy() == want).all(), (rate, n)
        if n in (1, enc.k // 8):
            # host memory with rows wider than 81 bytes: the padding comes back untouched
            out = np.full((3, 96), 0xA5, np.uint8)
            enc.encode_batch(pay, out=out)
            assert (out[:, :81] == want).all() and (out[:, 81:] == 0xA5).all()
            # device memory, padded payload and coded rows
            wide = torch.zeros((3, n + 7), dtype=torch.uint8, device="cuda")
            wide[:, :n] = torch.from_numpy(pay).cuda()
            dout = torch.full((3, 100), 7, dtype=torch.uint8, device="cuda")
            enc.encode_batch(wide[:, :n], out=dout)
            torch.cuda.synchronize()
            d = dout.cpu().numpy()
            assert (d[:, :81] == want).all() and (d[:, 81:] == 7).all()
    with pytest.raises(capi.PuError):
        enc.encode_batch(np.zeros((1, enc.k // 8 + 1), np.uint8))
    # B = 0: nothing to encode, in host and device memory
    assert enc.encode_batch(np.zeros((0, 5), np.uint8)).shape == (0, 81)
    assert tuple(enc.encode_batch(torch.zeros((0, 5), dtype=torch.uint8, device="cuda")).shape) == (0, 81)


@pytest.mark.parametrize("rate", RATES)
def test_frame_encode_batch_bit_identical(ctx, rate):
    import torch
    from projectultra_b200 import capi
    enc = capi.LdpcDecoder(ctx, rate)
    bpc = BPC[rate]
    rng = np.random.default_rng(100 + rate)
    for n in (1, 2, 5, 41, 255):
        nbytes = frame_size(bpc, n)
        assert enc.frame_codewords(nbytes) == n
        frames = rng.integers(0, 256, (3, nbytes), dtype=np.uint8)
        frames[1, : nbytes // 2] = 0
        want = np.stack([capi.frame_encode(rate, f).reshape(-1) for f in frames])
        assert want.shape == (3, n * 81)
        got, ncw = enc.frame_encode_batch(torch.from_numpy(frames).cuda())
        torch.cuda.synchronize()
        assert ncw == n and (got.cpu().numpy() == want).all(), (rate, n)
        out = np.full((3, n * 81 + 13), 0x5A, np.uint8)
        enc.frame_encode_batch(frames, out=out)
        assert (out[:, :n * 81] == want).all() and (out[:, n * 81:] == 0x5A).all(), (rate, n, "host")
        dout = torch.full((3, n * 81 + 40), 9, dtype=torch.uint8, device="cuda")
        wide = torch.zeros((3, nbytes + 3), dtype=torch.uint8, device="cuda")
        wide[:, :nbytes] = torch.from_numpy(frames).cuda()
        enc.frame_encode_batch(wide[:, :nbytes], out=dout)
        torch.cuda.synchronize()
        d = dout.cpu().numpy()
        assert (d[:, :n * 81] == want).all() and (d[:, n * 81:] == 9).all(), (rate, n, "device")
    # a frame that needs 256 codewords is refused; the query still answers
    big = frame_size(bpc, 256)
    assert enc.frame_codewords(big) == 256
    with pytest.raises(capi.PuError):
        enc.frame_encode_batch(np.zeros((1, big), np.uint8))
    # B = 0: the codeword count comes back, nothing is written
    empty, ncw = enc.frame_encode_batch(np.zeros((0, frame_size(bpc, 5)), np.uint8))
    assert ncw == 5 and empty.shape == (0, 5 * 81)


def raw_reference(llr, coded, n_bits, n_valid, index, bins, n_bins, strong):
    bits = np.unpackbits(coded[index], axis=1)[:, :n_bits].astype(bool)
    x = llr[:, :n_bits]
    valid = np.arange(n_bits)[None, :] < n_valid[:, None]
    zero = x == 0
    err = valid & ~zero & ((x < 0) != bits)
    out = np.zeros((n_bins, 4), np.int64)
    np.add.at(out[:, 0], bins, n_bits)
    np.add.at(out[:, 1], bins, (~valid | zero).sum(1))
    np.add.at(out[:, 2], bins, err.sum(1))
    np.add.at(out[:, 3], bins, (err & (np.abs(x) >= strong)).sum(1))
    return out


@pytest.mark.parametrize("n_bits,stride", [(648, 648), (3 * 648, 3 * 648 + 5)])
def test_count_raw_errors_matches_numpy(ctx, n_bits, stride):
    import torch
    from projectultra_b200 import capi
    rng = np.random.default_rng(n_bits)
    B, P, n_bins, strong = 5000, 37, 23, 10.0
    llr = (rng.normal(0, 6, (B, stride))).astype(np.float32)
    special = np.array([0.0, -0.0, 10.0, -10.0, np.nextafter(np.float32(10), np.float32(0)), -np.nextafter(np.float32(10), np.float32(0)),
                        np.nextafter(np.float32(10), np.float32(20)), -np.nextafter(np.float32(10), np.float32(20)), 1e-30, -1e-30], np.float32)
    pick = rng.random((B, stride)) < 0.2
    llr[pick] = special[rng.integers(0, len(special), pick.sum())]
    llr[5] = -0.0
    coded = rng.integers(0, 256, (P, (n_bits + 7) // 8 + 3), dtype=np.uint8)
    index = rng.integers(0, P, B).astype(np.uint32)
    bins = np.sort(rng.integers(0, n_bins, B)).astype(np.uint32)      # runs of one bin, as in a sweep batch
    bins[::97] = rng.integers(0, n_bins, len(bins[::97]))                # and stray rows
    n_valid = np.full(B, n_bits, np.int32)
    short = rng.random(B) < 0.1
    n_valid[short] = rng.integers(-5, n_bits, short.sum())
    n_valid[7] = n_bits + 100
    want = raw_reference(llr, coded, n_bits, np.clip(n_valid, 0, n_bits), index, bins, n_bins, strong)
    dev = lambda a, dt=None: torch.from_numpy(a.view(dt) if dt else a).cuda()
    d_llr, d_coded, d_idx, d_bins, d_nv = dev(llr), dev(coded), dev(index, np.int32), dev(bins, np.int32), dev(n_valid)
    # one launch
    c = torch.zeros((n_bins, 4), dtype=torch.int64, device="cuda")
    capi.count_raw_errors(ctx, d_llr, d_coded, c, n_bits, d_nv, d_idx, d_bins, strong)
    torch.cuda.synchronize()
    got = c.cpu().numpy()
    assert (got == want).all(), (got - want)[np.any(got != want, axis=1)]
    assert want[:, 1].sum() > 0 and want[:, 3].sum() > 0 and want[:, 2].sum() > want[:, 3].sum()
    # several launches on slices of the batch accumulate to the same table
    c.zero_()
    for a, b in ((0, 1), (1, 1000), (1000, 4321), (4321, B)):
        capi.count_raw_errors(ctx, d_llr[a:b], d_coded, c, n_bits, d_nv[a:b], d_idx[a:b], d_bins[a:b], strong)
    torch.cuda.synchronize()
    assert (c.cpu().numpy() == want).all()
    # no n_valid, no gather, no bins: every row counts in full against its own coded row, into row 0
    c1 = torch.zeros((1, 4), dtype=torch.int64, device="cuda")
    rows = rng.integers(0, 256, (B, (n_bits + 7) // 8), dtype=np.uint8)
    capi.count_raw_errors(ctx, d_llr, dev(rows), c1, n_bits, strong=strong)
    torch.cuda.synchronize()
    ref = raw_reference(llr, rows, n_bits, np.full(B, n_bits), np.arange(B), np.zeros(B, np.int64), 1, strong)
    assert (c1.cpu().numpy() == ref).all()


# ---------------------------------------------------------------- the sweep driver against LinkSim / FrameLinkSim (pool path)
def cfg_m1(capi, rate=R.R1_2, mod=R.DQPSK):
    return capi.ModemConfig.from_buffer_copy(bytes(R.config_m1(mod, rate)))


def mixed_table(capi):
    mc = capi.mcdpsk_config(8, 2)
    return [capi.sweep_mode(capi.WF_OFDM, cfg_m1(capi), R.R1_2, 40, "awgn", -3, 1.5, 3),
            capi.sweep_mode(capi.WF_OFDM, cfg_m1(capi), R.R1_2, 40, "moderate", 2, 3, 3, precision="fast", interleave_bps=60),
            capi.sweep_mode(capi.WF_OFDM_CHIRP, cfg_m1(capi, R.R1_4), R.R1_4, 20, "good", 20, 5, 2, peak=0.5, precision="fast"),
            capi.sweep_mode(capi.WF_DPSK_ACQ, capi.dpsk_config(1, 384), R.R1_4, 20, "awgn", -4, 4, 3, peak=0.5, lead_samples=0),
            capi.sweep_mode(capi.WF_MCDPSK_CHIRP, mc, R.R1_2, 40, "moderate", 0, 5, 3, interleave_bps=16, peak=0.5, lead_samples=480,
                            tail_samples=2400),
            capi.sweep_mode(capi.WF_OFDM, cfg_m1(capi), R.R1_2, 0, "good", 0, 3, 3, precision="fast", frame_payload_bytes=60, interleave_bps=60),
            capi.sweep_mode(capi.WF_OFDM_CHIRP, cfg_m1(capi), R.R1_2, 0, "moderate", 2, 3, 3, precision="fast", frame_payload_bytes=100,
                            interleave_bps=60, peak=0.5, lead_samples=480, tail_samples=2400),
            # interleaved and without tail silence: rows short of soft bits behind the deinterleaver (the driver maps each decoder position
            # back through the interleaver's step, LinkSim zeroes the undelivered bits through the permutation table)
            capi.sweep_mode(capi.WF_MCDPSK_CHIRP, mc, R.R1_2, 40, "moderate", 20, 5, 2, interleave_bps=16, peak=0.5),
            capi.sweep_mode(capi.WF_OFDM_CHIRP, cfg_m1(capi, R.R1_4), R.R1_4, 20, "good", 20, 5, 2, peak=0.5, precision="fast", interleave_bps=60),
            capi.sweep_mode(capi.WF_OFDM_CHIRP, cfg_m1(capi), R.R1_2, 0, "good", 20, 5, 2, precision="fast", frame_payload_bytes=100,
                            interleave_bps=60, peak=0.5)]


def linksim_tables(ctx, sw, mi, trials):
    """The driver's (mode, SNR point, trial) grid through LinkSim / FrameLinkSim with its pool and seeds: (counters, raw)."""
    import torch
    from projectultra_b200 import capi, linksim
    m = sw.modes[mi]
    pool = sw.desc.pool
    payloads = np.stack([sw.payload(mi, i) for i in range(pool)])
    chan = [k for k, v in capi.CHANNELS.items() if v == m.channel][0]
    chirp = m.waveform in (capi.WF_OFDM_CHIRP, capi.WF_MCDPSK_CHIRP)
    kw = dict(precision="fast" if m.precision else "exact", payloads=payloads, peak=m.peak or None, code_rate=m.code_rate, pool=pool,
              interleave_bps=m.interleave_bps)
    if chirp:
        kw.update(layout="chirp", lead_samples=m.lead_samples, tail_samples=m.tail_samples)
    if m.frame_payload_bytes:
        sim = linksim.FrameLinkSim(ctx, m.ofdm, chan, payload_bytes=m.frame_payload_bytes, **kw)
    else:
        cfg = m.ofdm if m.waveform <= capi.WF_OFDM_CHIRP else m.dpsk if m.waveform <= capi.WF_DPSK_ACQ else m.mcdpsk
        if m.waveform == capi.WF_DPSK_ACQ:
            kw.update(acquire=True)
        sim = linksim.LinkSim(ctx, cfg, chan, payload_bytes=m.payload_bytes, **kw)
    snrs = m.snr_points
    si = np.repeat(np.arange(len(snrs), dtype=np.int64), trials)
    tr = np.tile(np.arange(trials, dtype=np.int64), len(snrs))
    c = torch.zeros((len(snrs), 6), dtype=torch.int64, device="cuda")
    raw = torch.zeros((len(snrs), 4), dtype=torch.int64, device="cuda")
    sim.run_batch(sim.make_batch(snrs, si, tr, base_seed=0xB200 | (mi << 16)), c, raw=raw)      # (mode << 56) of the driver's seed rule
    torch.cuda.synchronize()
    return c.cpu().numpy().astype(np.uint64), raw.cpu().numpy().astype(np.uint64)


def test_driver_raw_table_matches_linksim(ctx):
    from projectultra_b200 import capi, linksim
    trials = 64
    modes = mixed_table(capi)
    sw = capi.Sweep(modes, trials_per_point=trials, block_trials=32, pool=8)
    plain, _ = sw.run(ctx)
    counters, st, raw = sw.run(ctx, raw=True)
    assert st.units_run == sw.n_units
    assert (counters == plain).all()                     # the unfused PU_WF_OFDM path decodes the same
    at = 0
    for mi, m in enumerate(modes):
        want_c, want_r = linksim_tables(ctx, sw, mi, trials)
        got_c, got_r = counters[at:at + m.n_snr], raw[at:at + m.n_snr]
        assert (got_c == want_c).all(), (mi, got_c.tolist(), want_c.tolist())
        assert (got_r == want_r).all(), (mi, got_r.tolist(), want_r.tolist())
        n_cw = got_c[0, 3] // trials if m.frame_payload_bytes else 1
        assert (got_r[:, 0] == trials * 648 * n_cw).all()
        at += m.n_snr
    rows = linksim.summarize(counters, [0.0] * sw.n_points, raw)
    print("raw BER:", [round(r["raw_ber"], 4) for r in rows])
    print("erasure rate:", [round(r["erasure_rate"], 4) for r in rows])
    print("strong error share:", [round(r["strong_error_share"], 3) for r in rows])
    assert raw[6:8, 1].sum() > 0                         # OFDM_CHIRP without tail silence: the last symbol is missing
    assert raw[0, 2] > raw[2, 2]                         # AWGN DQPSK: fewer raw errors up the grid
    assert (raw[8:11, 3] == 0).all()                     # single-carrier DPSK soft bits stop at 5
    # short interleaved rows: some soft bits missing, not all (the erasures come from the permutation, not from whole rows)
    assert (raw[20:26, 1] > 0).all() and (raw[20:26, 1] < raw[20:26, 0]).all() and (raw[20:26, 2] > 0).all(), raw[20:26].tolist()


def fresh_table(capi, fresh):
    mc = capi.mcdpsk_config(8, 2)
    return [capi.sweep_mode(capi.WF_OFDM, cfg_m1(capi), R.R1_2, 40, "awgn", -4, 1, 4, precision="fast", fresh_payloads=fresh),
            capi.sweep_mode(capi.WF_MCDPSK, mc, R.R1_2, 40, "moderate", 0, 3, 3, peak=0.5, interleave_bps=16, fresh_payloads=fresh),
            capi.sweep_mode(capi.WF_OFDM_CHIRP, cfg_m1(capi), R.R1_2, 0, "good", 2, 3, 3, precision="fast", frame_payload_bytes=100, peak=0.5,
                            lead_samples=480, tail_samples=2400, fresh_payloads=fresh)]


def per_frame_fractions(ctx, capi, modes, trials, d):
    """A raw run of one-trial work units with a manifest: (raw bit errors / non-erased soft bits of every frame [points, trials], raw table)."""
    sw = capi.Sweep(modes, trials_per_point=trials, block_trials=1, pool=32, manifest_dir=d, run_id=1)
    _, _, table = sw.run(ctx, raw=True)
    first = np.cumsum([0] + [m.n_snr for m in modes])
    f = np.full((sw.n_points, trials), np.nan)
    for name in os.listdir(d):
        for line in open(os.path.join(d, name)):
            if line.startswith("#"):
                continue
            v = [int(x) for x in line.split()[:11]]
            m, s, t0, _ = sw.unit(v[0])
            f[first[m] + s, t0] = v[9] / max(v[7] - v[8], 1)
    assert not np.isnan(f).any()
    return f, table


def test_fresh_raw_counts_match_the_pool_and_resume(ctx, tmp_path):
    from projectultra_b200 import capi
    trials = 512
    kw = dict(trials_per_point=trials, block_trials=128, pool=32)
    pool_c, _, pool_r = capi.Sweep(fresh_table(capi, False), **kw).run(ctx, raw=True)
    fresh_c, _, fresh_r = capi.Sweep(fresh_table(capi, True), **kw).run(ctx, raw=True)
    plain_c, _ = capi.Sweep(fresh_table(capi, True), **kw).run(ctx)
    assert (plain_c == fresh_c).all()
    again = capi.Sweep(fresh_table(capi, True), **kw).run(ctx, raw=True)
    assert (again[0] == fresh_c).all() and (again[2] == fresh_r).all()
    parts = [capi.Sweep(fresh_table(capi, True), rank=r, world=2, **kw).run(ctx, raw=True) for r in range(2)]
    assert (parts[0][2] + parts[1][2] == fresh_r).all() and (parts[0][0] + parts[1][0] == fresh_c).all()
    assert (fresh_r[:, 0] == pool_r[:, 0]).all()
    # raw BER of fresh trials within the pool's spread.  The bits of one frame share its noise and fading, so the frame, not the bit, is
    # the independent trial: one-trial work units put every frame's raw counters in the manifest, and the per-frame error fractions give
    # each point's mean and its standard error (sample variance over the frames)
    fp, tp = per_frame_fractions(ctx, capi, fresh_table(capi, False), trials, str(tmp_path / "frames_pool"))
    ff, tf = per_frame_fractions(ctx, capi, fresh_table(capi, True), trials, str(tmp_path / "frames_fresh"))
    assert (tp == pool_r).all() and (tf == fresh_r).all()          # one-trial units: the same frames, the same totals
    mp, mf = fp.mean(1), ff.mean(1)
    se = np.sqrt(fp.var(1, ddof=1) / trials + ff.var(1, ddof=1) / trials)
    print("raw BER per frame, pool :", mp.round(4).tolist())
    print("raw BER per frame, fresh:", mf.round(4).tolist())
    print("standard error of the difference:", se.round(5).tolist())
    assert mp[0] > 0.01 and (np.abs(mp - mf) <= 5 * se).all(), ((mp - mf) / np.maximum(se, 1e-12)).round(2).tolist()
    # an interrupted raw run resumes from its manifest to the uninterrupted totals
    d = str(tmp_path / "raw")
    _, s1, _ = capi.Sweep(fresh_table(capi, True), manifest_dir=d, max_units=5, run_id=1, **kw).run(ctx, raw=True)
    assert s1.units_run == 5
    tot_c, tot_r = np.zeros_like(fresh_c), np.zeros_like(fresh_r)
    for r in range(2):
        c, st, rr = capi.Sweep(fresh_table(capi, True), manifest_dir=d, rank=r, world=2, run_id=2, **kw).run(ctx, raw=True)
        assert st.units_resumed == 5
        tot_c += c
        tot_r += rr
    assert (tot_c == fresh_c).all() and (tot_r == fresh_r).all()
    # a raw run and a plain run never resume from each other's manifests
    with pytest.raises(capi.PuError):
        capi.Sweep(fresh_table(capi, True), manifest_dir=d, run_id=3, **kw).run(ctx)
    p = str(tmp_path / "plain")
    capi.Sweep(fresh_table(capi, True), manifest_dir=p, max_units=2, run_id=1, **kw).run(ctx)
    with pytest.raises(capi.PuError):
        capi.Sweep(fresh_table(capi, True), manifest_dir=p, run_id=2, **kw).run(ctx, raw=True)


def test_raw_ber_physical_sanity(ctx):
    from projectultra_b200 import capi
    mc = capi.mcdpsk_config(8, 2)
    modes = [capi.sweep_mode(capi.WF_OFDM, cfg_m1(capi), R.R1_2, 40, "awgn", -30, 2, 31, precision="fast"),
             capi.sweep_mode(capi.WF_MCDPSK, mc, R.R1_2, 40, "awgn", -30, 2, 31, peak=0.5)]
    trials = 256
    _, _, raw = capi.Sweep(modes, trials_per_point=trials, block_trials=256, pool=16).run(ctx, raw=True)
    ber = raw[:, 2] / np.maximum(raw[:, 0] - raw[:, 1], 1)
    print("raw BER OFDM   :", ber[:31].round(4).tolist())
    print("raw BER MC-DPSK:", ber[31:].round(4).tolist())
    for b in (ber[:31], ber[31:]):
        assert 0.45 <= b[0] <= 0.55 and b[-1] == 0.0
        # non-increasing over the grid within the spread of a frame-correlated count (sqrt(ber / trials) per point, generous)
        spread = 3 * np.sqrt(np.maximum(b[:-1], 1e-4) / trials)
        assert (b[1:] <= b[:-1] + spread).all()


def test_acquired_codeword_short_of_soft_bits_shows_erasures(ctx):
    from projectultra_b200 import capi
    m1 = cfg_m1(capi, R.R1_4)
    rate = {}
    for tail in (0, 2400):
        modes = [capi.sweep_mode(capi.WF_OFDM_CHIRP, m1, R.R1_4, 20, "good", 25, 5, 2, peak=0.5, precision="fast",
                                 lead_samples=480 if tail else 0, tail_samples=tail, fresh_payloads=True)]
        _, _, raw = capi.Sweep(modes, trials_per_point=128, block_trials=128, pool=8).run(ctx, raw=True)
        rate[tail] = raw[:, 1] / raw[:, 0]
    print("erasure rate without / with tail silence:", rate[0].tolist(), rate[2400].tolist())
    assert (rate[0] > 0.01).all() and (rate[2400] * 10 <= rate[0]).all()
