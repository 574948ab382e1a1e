"""Raw (pre-decoder) counts of real demodulator output against the plain-C oracle: on identical channel outputs (LinkSim.make_rx), the raw
table LinkSim.receive_count accumulates from the GPU's soft bits (pu_count_raw_errors) equals a numpy count of the oracle's soft bits for the
same frames, against the oracle's own encoding of the payloads sent.  Exact for 512-FFT DQPSK presynced (exact precision, with and without
the fused deinterleaver), single-carrier DPSK and MC-DPSK with genie timing (MC-DPSK also behind the deinterleaver); for 1024-FFT 32QAM
pilots/4 exact on every frame whose LLR words are identical (the LLR test lets the others differ within 1e-4), and everywhere the hard
decisions and erasures agree wherever the LLRs agree within that tolerance."""
import numpy as np
import pytest

import oracleapi as O
import refapi as R
from test_ofdm_gpu import llr_mismatches

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from projectultra_b200 import capi
    c = capi.Context(0)
    yield c
    c.close()


def numpy_counts(llr, coded, strong=10.0):
    """Per frame {soft_bits, erasures, bit_errors, strong_errors} of soft bits llr [B, 648] against coded [B, 81] (bits MSB first)."""
    bits = np.unpackbits(coded, axis=1)[:, :648].astype(bool)
    x = llr[:, :648]
    zero = x == 0
    err = ~zero & ((x < 0) != bits)
    return np.stack([np.full(len(x), 648), zero.sum(1), err.sum(1), (err & (np.abs(x) >= strong)).sum(1)], axis=1).astype(np.int64)


def by_bin(per_frame, bins, n_bins):
    out = np.zeros((n_bins, 4), np.int64)
    np.add.at(out, bins, per_frame)
    return out


def run(ctx, cfg, oracle_llr, chan, snrs, trials, rate, nbytes, deint_bps=0, **kw):
    """GPU raw table, GPU soft bits, oracle soft bits (decoder order) and the oracle's codewords of the frames of one batch."""
    import torch
    from projectultra_b200 import linksim
    sim = linksim.LinkSim(ctx, cfg, chan, payload_bytes=nbytes, pool=8, code_rate=rate, interleave_bps=deint_bps, **kw)
    si = np.repeat(np.arange(len(snrs)), trials)
    tr = np.tile(np.arange(trials), len(snrs))
    batch = sim.make_batch(snrs, si, tr)
    rx = sim.make_rx(batch)
    counters = torch.zeros((len(snrs), 6), dtype=torch.int64, device="cuda")
    raw = torch.zeros((len(snrs), 4), dtype=torch.int64, device="cuda")
    sim.receive_count(batch, rx, counters, raw=raw)
    gpu = sim.demod_llr(rx)[:, :648].cpu().numpy()
    torch.cuda.synchronize()
    rx_h = rx.cpu().numpy()
    ref = np.ascontiguousarray(oracle_llr(rx_h)[:, :648], np.float32)
    if deint_bps:
        ref = np.stack([O.channel_interleave(deint_bps, r.copy(), inverse=True) for r in ref]).astype(np.float32)
    coded = np.stack([O.ldpc_encode(rate, sim.payloads[i]) for i in batch["host"]["tx_index"]])
    return raw.cpu().numpy(), gpu, ref, coded, si, sim


def check_signs(gpu, ref):
    """Wherever the soft bits agree within the LLR tests' tolerance, hard decision and erasure agree too."""
    close = np.ones(gpu.size, bool)
    close[llr_mismatches(gpu.ravel(), ref.ravel())] = False
    g, r = gpu.ravel()[close], ref.ravel()[close]
    assert ((g < 0) == (r < 0)).all() and ((g == 0) == (r == 0)).all()
    return close.mean()


@pytest.mark.parametrize("deint", [False, True])
def test_ofdm_dqpsk_exact_presynced(ctx, deint):
    from projectultra_b200 import capi
    cfg = R.config_m1(R.DQPSK, R.R1_2)
    ccfg = capi.ModemConfig.from_buffer_copy(bytes(cfg))
    bps = 2 * capi.OfdmDemodulator(ctx, ccfg).n_data if deint else 0
    snrs = (-4.0, -1.0, 2.0, 6.0)
    raw, gpu, ref, coded, si, sim = run(ctx, ccfg, lambda x: O.ofdm_presynced_batch(cfg, x, 648)[0], "awgn", snrs, 24, R.R1_2, 40,
                                        deint_bps=bps, precision="exact")
    assert sim.ofdm.last_kernel == "ofdm_diff512_kernel"
    per_gpu, per_ref = numpy_counts(gpu, coded), numpy_counts(ref, coded)
    assert (raw == by_bin(per_gpu, si, len(snrs))).all()          # the kernel on real demodulator output
    assert (raw == by_bin(per_ref, si, len(snrs))).all(), (raw.tolist(), by_bin(per_ref, si, len(snrs)).tolist())
    check_signs(gpu, ref)
    print("DQPSK deint=%s raw BER" % deint, (raw[:, 2] / raw[:, 0]).round(4).tolist(), "words identical %.5f" %
          (gpu.view(np.uint32) == ref.view(np.uint32)).mean())
    assert raw[0, 2] > raw[-1, 2]


def test_sc_dpsk_genie(ctx):
    from projectultra_b200 import capi
    cfg = capi.dpsk_config(1, 384)
    snrs = (-6.0, 0.0, 8.0)
    data_start = 39 * 384
    raw, gpu, ref, coded, si, _ = run(ctx, cfg, lambda x: np.stack([O.dpsk_demod_soft(1, 384, f, data_start, 1)[:648] for f in x]),
                                      "poor", snrs, 8, R.R1_4, 20, peak=0.5)
    assert (gpu.view(np.uint32) == ref.view(np.uint32)).all()
    assert (raw == by_bin(numpy_counts(ref, coded), si, len(snrs))).all()
    assert (raw[:, 3] == 0).all() and raw[0, 2] > 0                  # soft bits stop at 5: no strong errors


@pytest.mark.parametrize("bps", [0, 16])
def test_mcdpsk_genie(ctx, bps):
    from projectultra_b200 import capi
    cfg = capi.mcdpsk_config(8, 2)
    snrs = (-2.0, 4.0, 12.0)
    raw, gpu, ref, coded, si, _ = run(ctx, cfg, lambda x: np.stack([O.mcdpsk_demod_soft(8, f, bits=2)[0][:648] for f in x]),
                                      "good", snrs, 16, R.R1_2, 40, deint_bps=bps)
    assert (gpu.view(np.uint32) == ref.view(np.uint32)).all()
    assert (raw == by_bin(numpy_counts(ref, coded), si, len(snrs))).all()
    assert raw[0, 2] > raw[-1, 2]


def test_ofdm_32qam_pilots(ctx):
    from projectultra_b200 import capi
    cfg = R.config_m3(R.QAM32, R.R3_4)
    snrs = (8.0, 12.0, 16.0, 24.0)
    raw, gpu, ref, coded, si, _ = run(ctx, capi.ModemConfig.from_buffer_copy(bytes(cfg)), lambda x: O.ofdm_presynced_batch(cfg, x, 648)[0],
                                      "good", snrs, 24, R.R3_4, 60)
    per_gpu, per_ref = numpy_counts(gpu, coded), numpy_counts(ref, coded)
    assert (raw == by_bin(per_gpu, si, len(snrs))).all()
    same = (gpu.view(np.uint32) == ref.view(np.uint32)).all(axis=1)
    print("32QAM: frames with identical LLR words %d / %d" % (same.sum(), len(same)))
    assert same.sum() > 0 and (per_gpu[same] == per_ref[same]).all()
    frac = check_signs(gpu, ref)
    assert frac > 0.999
    # frames whose soft bits all agree within the tolerance have the same erasures and bit errors
    within = ~np.isin(np.arange(len(gpu)), np.unique(llr_mismatches(gpu.ravel(), ref.ravel()) // 648))
    assert (per_gpu[within, 1:3] == per_ref[within, 1:3]).all()
