"""Host logic of ChannelInterleaver in the sweep driver (pu_sweep_mode.interleave_bps, csrc/sweep.cu) without a GPU: which waveforms may
interleave, in codeword and frame mode, and a table without the field enumerating and partitioning exactly as before."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def m1(capi):
    return capi.ModemConfig(48000, 1500, 512, 30, 1, 4, 2, 0, capi.DQPSK, capi.R1_2, 40.0, 0.0)


def unit_count(capi, modes):
    import ctypes as C
    sw = object.__new__(capi.Sweep)          # the description only: Sweep() refuses an invalid table before we can look at it
    sw.modes = list(modes)
    sw._arr = (capi.SweepMode * len(sw.modes))(*sw.modes)
    sw.desc = capi.SweepDesc(sw._arr, len(sw.modes), 64, 4096, 4096, 50, 0xB200, 0, 1, 0, None, 0, 0)
    f = capi.lib().pu_sweep_unit_count
    f.restype = C.c_uint64
    return int(f(C.byref(sw.desc)))


def test_single_carrier_dpsk_rows_cannot_interleave():
    from projectultra_b200 import capi
    ok = capi.sweep_mode(capi.WF_OFDM, m1(capi), capi.R1_2, 40, "awgn", 0, 1, 3, interleave_bps=60)
    assert unit_count(capi, [ok]) == 3
    for wf in (capi.WF_DPSK, capi.WF_DPSK_ACQ):
        plain = capi.sweep_mode(wf, capi.dpsk_config(1, 384), capi.R1_4, 20, "awgn", 0, 1, 3)
        assert unit_count(capi, [ok, plain]) == 6
        bad = capi.sweep_mode(wf, capi.dpsk_config(1, 384), capi.R1_4, 20, "awgn", 0, 1, 3, interleave_bps=2)
        assert unit_count(capi, [ok, bad]) == 0
        with pytest.raises(capi.PuError):
            capi.Sweep([ok, bad], trials_per_point=4096)


def test_ofdm_and_mcdpsk_rows_interleave_in_codeword_and_frame_mode():
    from projectultra_b200 import capi
    mc = capi.mcdpsk_config(8, 2)
    for bps in (1, 60, 118, 700):
        modes = [capi.sweep_mode(wf, m1(capi), capi.R1_2, 40, "good", 0, 1, 2, interleave_bps=bps)
                 for wf in (capi.WF_OFDM, capi.WF_OFDM_SC, capi.WF_OFDM_CHIRP)]
        modes += [capi.sweep_mode(wf, m1(capi), capi.R1_2, 0, "good", 0, 1, 2, frame_payload_bytes=200, interleave_bps=bps)
                  for wf in (capi.WF_OFDM, capi.WF_OFDM_SC, capi.WF_OFDM_CHIRP)]
        modes += [capi.sweep_mode(wf, mc, capi.R1_2, 40, "poor", 0, 1, 2, interleave_bps=bps) for wf in (capi.WF_MCDPSK, capi.WF_MCDPSK_CHIRP)]
        assert unit_count(capi, modes) == 16
        sw = capi.Sweep(modes, trials_per_point=8192, block_trials=4096)
        assert sw.n_units == 32 and sw.n_points == 16
    # MC-DPSK frame modes stay invalid, interleaved or not
    assert unit_count(capi, [capi.sweep_mode(capi.WF_MCDPSK, mc, capi.R1_2, 40, "awgn", 0, 1, 2, frame_payload_bytes=100, interleave_bps=16)]) == 0


def table(capi, interleave):
    q16 = capi.ModemConfig(48000, 1500, 512, 30, 1, 4, 2, 1, capi.QAM16, capi.R1_2, 40.0, 0.0)
    il = (lambda n: dict(interleave_bps=n)) if interleave else (lambda n: {})
    return [capi.sweep_mode(capi.WF_OFDM, m1(capi), capi.R1_2, 40, "awgn", -4, 1, 13, precision="fast", **il(60)),
            capi.sweep_mode(capi.WF_OFDM, q16, capi.R1_2, 0, "good", 6, 2, 12, frame_payload_bytes=1000, **il(112)),
            capi.sweep_mode(capi.WF_OFDM_CHIRP, m1(capi), capi.R1_2, 0, "good", 0, 2, 12, peak=0.5, lead_samples=480, tail_samples=2400,
                            frame_payload_bytes=200, **il(60)),
            capi.sweep_mode(capi.WF_DPSK_ACQ, capi.dpsk_config(1, 384), capi.R1_4, 20, "poor", -11, 2, 15, peak=0.5),
            capi.sweep_mode(capi.WF_MCDPSK, capi.mcdpsk_config(8, 2), capi.R1_2, 40, "moderate", -2, 2, 8, **il(16))]


def test_a_table_without_the_field_enumerates_and_partitions_as_before():
    """The field is appended; 0 is the zero-initialised default.  Interleaving changes what a unit computes, not how many units there
    are, what they cost or who runs them."""
    from projectultra_b200 import capi
    plain = capi.Sweep(table(capi, False), trials_per_point=4096, block_trials=1024, world=2)
    assert all(m.interleave_bps == 0 for m in plain.modes)
    assert capi.sweep_mode(capi.WF_OFDM, m1(capi), capi.R1_2, 40, "awgn", 0, 1, 3).interleave_bps == 0
    inter = capi.Sweep(table(capi, True), trials_per_point=4096, block_trials=1024, world=2)
    assert (plain.n_units, plain.n_points) == (inter.n_units, inter.n_points) == (4 * 60, 60)
    (o1, c1), (o2, c2) = plain.partition(), inter.partition()
    assert (o1 == o2).all() and (c1 == c2).all()
    assert [plain.unit(u) for u in range(plain.n_units)] == [inter.unit(u) for u in range(inter.n_units)]
    load = np.bincount(o1, weights=c1, minlength=2)
    assert abs(load[0] / load.sum() - 0.5) < 0.05
    assert (plain.payload(1, 3) == inter.payload(1, 3)).all()


def test_abi_size_of_the_mode_includes_the_new_field():
    import ctypes as C
    from projectultra_b200 import capi
    out = (C.c_uint32 * 8)()
    capi.lib().pu_abi_sizes(out)
    assert out[4] == C.sizeof(capi.SweepMode) and capi.SweepMode.interleave_bps.offset == C.sizeof(capi.SweepMode) - 4
