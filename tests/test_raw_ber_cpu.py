"""Host side of the raw (pre-decoder) bit error counts: the counter names, linksim.summarize's raw columns and the exported entry points."""
import numpy as np
import pytest


@pytest.fixture(scope="module")
def capi():
    from projectultra_b200 import build, capi
    build.build()
    return capi


def test_raw_counter_names():
    from projectultra_b200 import linksim
    assert linksim.RAW_COUNTER_NAMES == ("soft_bits", "erasures", "bit_errors", "strong_errors")
    assert linksim.RAW_STRONG == 10.0


def test_summarize_raw_columns():
    from projectultra_b200 import linksim
    counters = np.array([[100, 40, 900, 32000, 30, 4000], [100, 0, 0, 32000, 0, 300]], np.uint64)
    raw = np.array([[64800, 800, 12800, 12544], [64800, 0, 0, 0]], np.uint64)
    rows = linksim.summarize(counters, [-2.0, 10.0], raw)
    assert rows[0]["raw_ber"] == 12800 / 64000 and rows[0]["erasure_rate"] == 800 / 64800
    assert rows[0]["strong_error_share"] == 12544 / 12800
    assert rows[1]["raw_ber"] == 0.0 and rows[1]["strong_error_share"] == 0.0
    assert rows[0]["fer"] == 0.4 and "fer_ci" in rows[0] and "raw_ber_ci" not in rows[0]
    # without a raw table the rows are what they were
    plain = linksim.summarize(counters, [-2.0, 10.0])
    assert all("raw_ber" not in r for r in plain)
    assert [{k: v for k, v in r.items() if k in plain[0]} for r in rows] == plain


def test_raw_entry_points_are_exported(capi):
    L = capi.lib()
    for name in ("pu_ldpc_encode_batch", "pu_frame_encode_batch", "pu_count_raw_errors", "pu_linksim_run_raw"):
        assert hasattr(L, name), name


@pytest.mark.parametrize("bps", [16, 60, 220])
def test_erase_undelivered_follows_the_deinterleaver(capi, bps):
    """A receiver that delivered n_valid soft bits (its order) leaves the rest undelivered; behind ChannelInterleaver::deinterleave (the
    oracle's) they sit elsewhere.  linksim.erase_undelivered must zero exactly those, whatever the undelivered entries held."""
    import torch
    import oracleapi as O
    from projectultra_b200 import linksim
    rng = np.random.default_rng(bps)
    n_cw, B = 3, 6
    delivered = rng.uniform(0.5, 10, (B, n_cw * 648)).astype(np.float32) * rng.choice([-1, 1], (B, n_cw * 648))
    n_valid = np.array([0, 1, 647, 648, 1000, n_cw * 648 + 5], np.int32)
    deint = lambda rows: np.stack([np.concatenate([O.channel_interleave(bps, r[c * 648:(c + 1) * 648].copy(), inverse=True) for c in range(n_cw)])
                                   for r in rows]).astype(np.float32)
    zeroed = delivered.copy()
    zeroed[np.arange(n_cw * 648)[None, :] >= n_valid[:, None]] = 0.0
    want = deint(zeroed)
    got = linksim.erase_undelivered(torch.from_numpy(deint(delivered)), torch.from_numpy(n_valid), n_cw * 648, bps).numpy()
    assert (got == want).all()
