"""Host logic of the sweep driver's frame modes (pu_sweep_mode.frame_payload_bytes, csrc/sweep.cu) without a GPU: which frame tables are
valid, the codeword count limit, the partitioner's cost of a frame and its balance on a mixed table, and the pool payloads."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def m1(capi, mod=None, pilots=0):
    return capi.ModemConfig(48000, 1500, 512, 30, 1, 4, 2, pilots, capi.DQPSK if mod is None else mod, capi.R1_2, 40.0, 0.0)


def unit_count(capi, modes, **kw):
    import ctypes as C
    sw = object.__new__(capi.Sweep)          # the description only: Sweep() refuses an invalid table before we can look at it
    sw.modes = list(modes)
    sw._arr = (capi.SweepMode * len(sw.modes))(*sw.modes)
    sw.desc = capi.SweepDesc(sw._arr, len(sw.modes), kw.get("pool", 64), kw.get("trials", 4096), 4096, 50, 0xB200, 0, 1, 0, None, 0, 0)
    f = capi.lib().pu_sweep_unit_count
    f.restype = C.c_uint64
    return int(f(C.byref(sw.desc)))


def bytes_for_codewords(bpc, n):
    """Largest payload whose DATA frame (payload + 19 bytes) needs exactly n codewords of bpc bytes (CW1+ carry bpc - 2)."""
    return bpc + (n - 1) * (bpc - 2) - 19


def test_frame_modes_are_validated_on_the_host():
    from projectultra_b200 import capi
    ok = capi.sweep_mode(capi.WF_OFDM, m1(capi), capi.R1_4, 0, "awgn", 0, 1, 3, frame_payload_bytes=200)
    assert unit_count(capi, [ok]) == 3                                        # payload_bytes is unused in frame modes: 0 is fine
    for wf in (capi.WF_OFDM_SC, capi.WF_OFDM_CHIRP):
        assert unit_count(capi, [capi.sweep_mode(wf, m1(capi), capi.R1_2, 0, "good", 0, 1, 2, frame_payload_bytes=1000)]) == 2
    bad = [capi.sweep_mode(capi.WF_DPSK, capi.dpsk_config(1, 384), capi.R1_4, 20, "awgn", 0, 1, 3, frame_payload_bytes=100),
           capi.sweep_mode(capi.WF_DPSK_ACQ, capi.dpsk_config(1, 384), capi.R1_4, 20, "awgn", 0, 1, 3, frame_payload_bytes=100),
           capi.sweep_mode(capi.WF_MCDPSK, capi.mcdpsk_config(8, 2), capi.R1_2, 40, "awgn", 0, 1, 3, frame_payload_bytes=100),
           capi.sweep_mode(capi.WF_MCDPSK_CHIRP, capi.mcdpsk_config(8, 2), capi.R1_2, 40, "awgn", 0, 1, 3, frame_payload_bytes=100),
           # R1/4: 20 bytes per codeword, 18 behind the {0xD5, index} prefix -> one byte more than 255 codewords carry
           capi.sweep_mode(capi.WF_OFDM, m1(capi), capi.R1_4, 0, "awgn", 0, 1, 3, frame_payload_bytes=bytes_for_codewords(20, 255) + 1),
           capi.sweep_mode(capi.WF_OFDM, m1(capi), capi.R5_6, 0, "awgn", 0, 1, 3, frame_payload_bytes=65536)]
    for b in bad:
        assert unit_count(capi, [ok, b]) == 0, (b.waveform, b.frame_payload_bytes)
        with pytest.raises(capi.PuError):
            capi.Sweep([ok, b], trials_per_point=4096)
    # the largest frame that still fits 255 codewords is valid
    edge = capi.sweep_mode(capi.WF_OFDM, m1(capi), capi.R1_4, 0, "awgn", 0, 1, 3, frame_payload_bytes=bytes_for_codewords(20, 255))
    assert unit_count(capi, [edge]) == 3
    # the codeword-mode rule is unchanged: payload_bytes 0 is only allowed in frame modes (checked when the mode is built), and a table
    # without frame modes enumerates as before
    assert unit_count(capi, [capi.sweep_mode(capi.WF_OFDM, m1(capi), capi.R1_2, 40, "awgn", 0, 1, 5)]) == 5


def mixed_table(capi):
    q16 = m1(capi, capi.QAM16, 1)
    m3 = capi.ModemConfig(48000, 1500, 1024, 59, 1, 0, 4, 1, capi.QAM32, capi.R3_4, 40.0, 0.0)
    return [capi.sweep_mode(capi.WF_OFDM, m1(capi), capi.R1_2, 40, "awgn", -4, 1, 13, precision="fast"),
            capi.sweep_mode(capi.WF_OFDM, m1(capi), capi.R1_2, 0, "awgn", -2, 1, 12, frame_payload_bytes=200),
            capi.sweep_mode(capi.WF_OFDM, q16, capi.R1_2, 0, "good", 6, 2, 12, frame_payload_bytes=1000),
            capi.sweep_mode(capi.WF_OFDM, m3, capi.R3_4, 0, "poor", 10, 2, 12, frame_payload_bytes=1000),
            capi.sweep_mode(capi.WF_OFDM_CHIRP, m1(capi), capi.R1_2, 0, "good", 0, 2, 12, peak=0.5, lead_samples=480, tail_samples=2400,
                            frame_payload_bytes=200),
            capi.sweep_mode(capi.WF_DPSK_ACQ, capi.dpsk_config(1, 384), capi.R1_4, 20, "poor", -11, 2, 15, peak=0.5),
            capi.sweep_mode(capi.WF_MCDPSK, capi.mcdpsk_config(8, 2), capi.R1_2, 40, "moderate", -2, 2, 8)]


def test_mixed_codeword_and_frame_table_splits_evenly_over_two_ranks():
    from projectultra_b200 import capi
    sw = capi.Sweep(mixed_table(capi), trials_per_point=4096, block_trials=1024, world=2)
    owner, cost = sw.partition()
    assert (owner < 2).all() and (cost > 0).all()
    load = np.bincount(owner, weights=cost, minlength=2)
    assert abs(load[0] / load.sum() - 0.5) < 0.05, load / load.sum()
    for r in range(2):                                                        # every rank computes the same assignment
        assert (capi.Sweep(mixed_table(capi), trials_per_point=4096, block_trials=1024, world=2, rank=r).partition()[0] == owner).all()


def test_a_frame_costs_its_length_and_codewords():
    from projectultra_b200 import capi
    modes = [capi.sweep_mode(capi.WF_OFDM, m1(capi), capi.R1_2, 40, "awgn", 0, 1, 1),
             capi.sweep_mode(capi.WF_OFDM, m1(capi), capi.R1_2, 0, "awgn", 0, 1, 1, frame_payload_bytes=200),
             capi.sweep_mode(capi.WF_OFDM, m1(capi), capi.R1_2, 0, "awgn", 0, 1, 1, frame_payload_bytes=1000)]
    _, cost = capi.Sweep(modes, trials_per_point=4096).partition()
    # R1/2: 219-byte frame = 6 codewords, 1019-byte frame = 27 codewords
    assert cost[0] * 4 < cost[1] < cost[0] * 7 and cost[1] * 3.5 < cost[2] < cost[1] * 5, cost.tolist()
    # a table's own per-trial cost is taken as it is
    modes[2].cost = 2.0
    _, c2 = capi.Sweep(modes, trials_per_point=4096).partition()
    assert c2[2] < cost[2]


def test_pool_payloads_of_frame_modes_have_the_frame_payload_length():
    from projectultra_b200 import capi
    sw = capi.Sweep(mixed_table(capi), trials_per_point=100)
    assert len(sw.payload(0, 3)) == 40 and len(sw.payload(1, 3)) == 200 and len(sw.payload(2, 3)) == 1000
    assert (sw.payload(2, 3)[:40] != sw.payload(0, 3)).any() and (sw.payload(2, 3) == sw.payload(2, 3)).all()
