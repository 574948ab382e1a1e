"""Host-memory batch calls against their own device paths: every PU_MEM_HOST entry point is run on the same seeded input once
with numpy arrays (staged through the context's pinned and device buffers, pu::HostStage in csrc/pu_ctx.cu) and once with CUDA
tensors whose outputs start zeroed, and every output must agree byte for byte.  Batches larger than one 64 MiB staging slab,
transmitter rows wider than a frame and an out-of-range pool index are covered as well."""
import ctypes as C

import numpy as np
import pytest

import refapi as R

pytestmark = pytest.mark.gpu

SENTINEL = np.uint32(0x7FC0BEEF)        # a NaN pattern in the padding of output rows: any write shows
SLAB = 64 << 20                         # staged row bytes per slab of the host calls


@pytest.fixture(scope="module")
def ctx():
    from projectultra_b200 import capi
    c = capi.Context(0)
    yield c
    c.close()


def dev(x):
    import torch
    return None if x is None else torch.from_numpy(np.ascontiguousarray(x)).cuda()


def same(host, device):
    """Both results (arrays or tuples of arrays, None where an output is absent) agree byte for byte."""
    import torch
    torch.cuda.synchronize()
    if not isinstance(host, tuple):
        host, device = (host,), (device,)
    assert len(host) == len(device)
    for i, (h, d) in enumerate(zip(host, device)):
        if h is None:
            assert d is None, i
            continue
        d = d.cpu().numpy() if isinstance(d, torch.Tensor) else np.asarray(d)
        h = np.asarray(h)
        assert h.dtype == d.dtype and h.shape == d.shape, (i, h.dtype, d.dtype, h.shape, d.shape)
        assert h.tobytes() == d.tobytes(), (i, np.flatnonzero(h.view(np.uint8) != d.view(np.uint8))[:8])


def noisy(rng, x, snr_db):
    p = float(np.mean(x.astype(np.float64) ** 2))
    return (x + rng.normal(0.0, np.sqrt(p / 10 ** (snr_db / 10)), x.shape)).astype(np.float32)


def wide(B, L, pad):
    return np.full((B, L + pad), SENTINEL, np.uint32).view(np.float32)


@pytest.fixture(scope="module")
def ofdm(ctx):
    from projectultra_b200 import capi
    cfg = R.config_m1(R.DQPSK, R.R1_2)
    dem = capi.OfdmDemodulator(ctx, cfg)
    enc = capi.LdpcDecoder(ctx, R.R1_2)
    yield dem, enc
    dem.close()
    enc.close()


def test_ofdm_tx_leaves_row_padding(ofdm):
    dem, enc = ofdm
    rng = np.random.default_rng(1)
    for layout in (0, 1):
        payload = rng.integers(0, 256, (5, 40), dtype=np.uint8)
        L = dem.tx_frame_len(enc, layout)
        h = dem.tx_batch(enc, payload, layout=layout, peak=0.5, out=wide(5, L, 37))
        d = dem.tx_batch(enc, dev(payload), layout=layout, peak=0.5, out=dev(wide(5, L, 37)))
        same(h, d)
        assert (h[:, L:].view(np.uint32) == SENTINEL).all()
        frames = rng.integers(0, 256, (3, 500), dtype=np.uint8)
        Lf = dem.frame_tx_batch(enc, frames, layout=layout)[0].shape[1]
        h, n = dem.frame_tx_batch(enc, frames, layout=layout, out=wide(3, Lf, 11))
        d, nd = dem.frame_tx_batch(enc, dev(frames), layout=layout, out=dev(wide(3, Lf, 11)))
        same(h, d)
        assert n == nd and (h[:, Lf:].view(np.uint32) == SENTINEL).all()
    # a batch of rows that takes more than one staging slab
    L = dem.tx_frame_len(enc, 0)
    B = SLAB // (4 * L + 40) + 5
    payload = rng.integers(0, 256, (B, 40), dtype=np.uint8)
    same(dem.tx_batch(enc, payload), dem.tx_batch(enc, dev(payload), out=dev(np.zeros((B, L), np.float32))))


def test_ofdm_receive_paths(ofdm):
    import torch
    dem, enc = ofdm
    rng = np.random.default_rng(2)
    payload = rng.integers(0, 256, (6, 40), dtype=np.uint8)
    tx = dem.tx_batch(enc, payload, layout=0)
    x = noisy(rng, tx, 8.0)
    B, L = x.shape
    n = dem.n_llr(L)
    z = lambda *s: torch.zeros(s, dtype=torch.float32, device="cuda")
    cfo = rng.uniform(-3, 3, B).astype(np.float32)
    same(dem.presynced_batch(x, llr_stride=n + 9), dem.presynced_batch(dev(x), llr_stride=n + 9, snr_db=z(B), final_cfo=z(B)))
    same(dem.presynced_batch(x, cfo_hz=cfo), dem.presynced_batch(dev(x), cfo_hz=dev(cfo), snr_db=z(B), final_cfo=z(B)))
    same(dem.presynced_batch(x, want_aux=False), dem.presynced_batch(dev(x), want_aux=False))
    same(dem.training_cfo_batch(x), dem.training_cfo_batch(dev(x)))
    # more frames than one staging slab holds
    big = noisy(rng, np.tile(tx, (SLAB // (4 * L * B) + 1, 1)), 6.0)
    same(dem.presynced_batch(big), dem.presynced_batch(dev(big), snr_db=z(len(big)), final_cfo=z(len(big))))
    # acquisition: Schmidl-Cox preamble frames behind silence
    sc = noisy(rng, np.concatenate([np.zeros((B, 1500), np.float32), dem.tx_batch(enc, payload, layout=1)], axis=1), 10.0)
    same(dem.acquire_batch(sc), dem.acquire_batch(dev(sc)))
    same(dem.process_batch(sc, llr_stride=700), dem.process_batch(dev(sc), llr_stride=700))


def test_ofdm_chirp_receive(ctx, ofdm):
    from projectultra_b200 import capi
    dem, enc = ofdm
    rng = np.random.default_rng(3)
    body = dem.tx_batch(enc, rng.integers(0, 256, (3, 40), dtype=np.uint8))
    chirp = capi.chirp_generate(48000.0, 0.0)
    x = np.stack([np.concatenate([np.zeros(300 + 700 * b, np.float32), chirp, body[b], np.zeros(1400 - 700 * b, np.float32)]) for b in range(3)])
    x = noisy(rng, x, 12.0)
    x[2] = noisy(rng, np.zeros_like(x[2]) + 0.01, 0.0)            # noise only: no detection, no soft bits
    same(dem.chirp_receive_batch(x, llr_stride=700), dem.chirp_receive_batch(dev(x), llr_stride=700))
    same(dem.chirp_receive_batch(x, want_llr=False), dem.chirp_receive_batch(dev(x), want_llr=False))


def psk_tx(fn, h, enc, payload, out, space):
    """pu_dpsk_tx_batch / pu_mcdpsk_tx_batch into rows of `out` (wider than a frame)."""
    from projectultra_b200 import capi
    n = C.c_size_t(0)
    capi.check(fn(h, enc._h, capi._ptr(payload), C.c_size_t(payload.shape[1]), C.c_size_t(payload.shape[1]), C.c_size_t(payload.shape[0]),
                  C.c_float(0.5), capi._ptr(out), C.c_size_t(out.shape[1]), C.byref(n), space, capi._stream(space)))
    return int(n.value)


def test_dpsk_paths(ctx):
    from projectultra_b200 import capi
    cfg = capi.dpsk_config(1, 384)
    dem = capi.DpskDemodulator(ctx, cfg)
    enc = capi.LdpcDecoder(ctx, R.R1_2)
    rng = np.random.default_rng(4)
    payload = rng.integers(0, 256, (4, 40), dtype=np.uint8)
    tx = dem.tx_batch(enc, payload)
    B, L = tx.shape
    h, d = wide(B, L, 29), dev(wide(B, L, 29))
    psk_tx(capi.lib().pu_dpsk_tx_batch, dem._h, enc, payload, h, capi.PU_MEM_HOST)
    psk_tx(capi.lib().pu_dpsk_tx_batch, dem._h, enc, dev(payload), d, capi.PU_MEM_DEVICE)
    same(h[:, :L], d[:, :L])
    assert (h[:, L:] == 0).all()                                  # host rows come back whole: zeros beyond the frame
    x = noisy(rng, np.concatenate([np.zeros((B, 2000), np.float32), tx], axis=1), 9.0)
    same(dem.receive_batch(x), dem.receive_batch(dev(x)))
    same(dem.receive_batch(x, want_llr=False), dem.receive_batch(dev(x), want_llr=False))
    ds = 39 * 384 + 2000
    cfo = rng.uniform(-2, 2, B).astype(np.float32)
    same(dem.demod_soft_batch(x, ds, est_cfo=cfo), dem.demod_soft_batch(dev(x), ds, est_cfo=dev(cfo)))
    dem.close()
    enc.close()


def test_mcdpsk_paths(ctx):
    from projectultra_b200 import capi
    cfg = capi.mcdpsk_config(8, 2)
    dem = capi.McDpskDemodulator(ctx, cfg)
    enc = capi.LdpcDecoder(ctx, R.R1_2)
    rng = np.random.default_rng(5)
    payload = rng.integers(0, 256, (4, 40), dtype=np.uint8)
    tx = dem.tx_batch(enc, payload)
    B, L = tx.shape
    h, d = wide(B, L, 13), dev(wide(B, L, 13))
    psk_tx(capi.lib().pu_mcdpsk_tx_batch, dem._h, enc, payload, h, capi.PU_MEM_HOST)
    psk_tx(capi.lib().pu_mcdpsk_tx_batch, dem._h, enc, dev(payload), d, capi.PU_MEM_DEVICE)
    same(h[:, :L], d[:, :L])
    assert (h[:, L:] == 0).all()
    x = noisy(rng, tx, 10.0)
    same(dem.demod_soft_batch(x, llr_stride=700), dem.demod_soft_batch(dev(x), llr_stride=700))
    cfo = np.array([0.0, 0.05, 0.4, -3.0], np.float32)
    same(dem.got_chirp_batch(x, cfo, llr_stride=700), dem.got_chirp_batch(dev(x), cfo, llr_stride=700))
    chirp = capi.chirp_generate(48000.0, 0.0)
    xc = noisy(rng, np.stack([np.concatenate([np.zeros(200 + 300 * b, np.float32), chirp, tx[b], np.zeros(1200 - 300 * b, np.float32)])
                              for b in range(B)]), 12.0)
    same(dem.chirp_receive_batch(xc, llr_stride=700), dem.chirp_receive_batch(dev(xc), llr_stride=700))
    dem.close()
    enc.close()


def test_channel_paths(ctx):
    from projectultra_b200 import capi, linksim
    rng = np.random.default_rng(6)
    P, L, B = 5, 3000, 7
    pool = rng.standard_normal((P, L)).astype(np.float32)
    idx = rng.integers(0, P, B).astype(np.uint32)
    std = rng.uniform(0.1, 0.5, B).astype(np.float32)
    seed = rng.integers(0, 2 ** 63, B, dtype=np.uint64)
    for name in ("awgn", "poor"):
        ch = linksim.channel_preset(name)
        same(linksim.channel_apply(ctx, ch, pool, idx, std, seed),
             linksim.channel_apply(ctx, ch, dev(pool), dev(idx), dev(std), dev(seed), rx=dev(np.zeros((B, L), np.float32))))
        same(linksim.channel_apply(ctx, ch, pool, None, std, seed),
             linksim.channel_apply(ctx, ch, dev(pool), None, dev(std), dev(seed), rx=dev(np.zeros((B, L), np.float32))))
    bad = idx.copy()
    bad[3] = P
    with pytest.raises(capi.PuError, match="invalid argument"):
        linksim.channel_apply(ctx, linksim.channel_preset("awgn"), pool, bad, std, seed)
    cfo = rng.uniform(-20, 20, B).astype(np.float32)
    same(linksim.channel_apply_cfo(ctx, pool[idx].copy(), cfo), linksim.channel_apply_cfo(ctx, dev(pool[idx]), dev(cfo)))


def test_decoders(ctx):
    from projectultra_b200 import capi
    rng = np.random.default_rng(7)
    enc = capi.LdpcDecoder(ctx, R.R1_2)
    kb = enc.info_bytes
    B = SLAB // (648 * 4) + 3                                     # more codewords than one staging slab holds
    llr = rng.normal(0.0, 4.0, (B, 700)).astype(np.float32)
    info = np.full((B, kb + 5), 0xAB, np.uint8)
    same(enc.decode_batch(llr, info=info), enc.decode_batch(dev(llr), info=dev(np.full((B, kb + 5), 0xAB, np.uint8)),
                                                            ok=dev(np.zeros(B, np.uint8)), iters=dev(np.zeros(B, np.int32))))
    assert (info[:, kb:] == 0xAB).all()
    for ncw in (1, 4):
        frames = rng.normal(1.5, 2.0, (6, ncw * 648)).astype(np.float32)
        same(enc.frame_decode_batch(frames, ncw), enc.frame_decode_batch(dev(frames), ncw))
    enc.close()


def test_tools_cfo(ctx):
    from projectultra_b200 import capi
    rng = np.random.default_rng(8)
    for n in (1000, 20000):
        cfo = capi.ToolsCfo(ctx, n, 7.5)
        x = wide(9, n, 21)
        x[:, :n] = rng.standard_normal((9, n)).astype(np.float32)
        d = dev(x)
        same(cfo.apply_batch(x), cfo.apply_batch(d))
        assert (x[:, n:].view(np.uint32) == SENTINEL).all()
        cfo.close()
