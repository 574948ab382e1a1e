"""Timing of ChannelInterleaver on the GPU: the batched deinterleaver (pu_llr_deinterleave_batch) and the transmitters with and without
pu_*_set_tx_interleave.

    python tools/interleave_bench.py [--out profiles/r2_interleave/interleave_bench.json]

Deinterleaver: CUDA events around 20 in-place calls on a device tensor [B, n_cw * 648] after 3 warm-up calls, at sizes of 0.5 to 2 GB
(4 to 16 times the 126 MB of L2, so every pass reads HBM); GB/s against the 8 bytes per soft bit the call must move (4 read, 4 written).
Transmitters: 20 calls of pu_frame_tx_batch (512-FFT DQPSK R1/2, 1 and 27 codewords per frame) and pu_mcdpsk_tx_batch (8 carriers DQPSK
R1/2) on fresh device payloads, interleaving off and on alternately, same inputs.  The card's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def timed(torch, fn, reps=20, warm=3):
    for _ in range(warm):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def bench_deinterleave(ctx, capi, torch):
    out = []
    for n_cw, rows in ((1, 200_000), (1, 800_000), (27, 8_000), (27, 30_000)):
        llr = torch.randn((rows, n_cw * 648), dtype=torch.float32, device="cuda")
        ms = timed(torch, lambda: capi.llr_deinterleave_batch(ctx, llr, n_cw, 60))
        n = rows * n_cw * 648
        r = dict(rows=rows, codewords_per_row=n_cw, gbytes=round(n * 4 / 1e9, 3), ms_per_call=round(ms, 3), gb_per_s=round(n * 8 / ms / 1e6, 1),
                 codewords_per_s=round(rows * n_cw / ms * 1e3))
        print("deinterleave", r, flush=True)
        out.append(r)
        del llr
    return out


def bench_tx(ctx, capi, torch, n_frames=4096):
    out = {}
    cfg = capi.ModemConfig(48000, 1500, 512, 30, 1, 4, 2, 0, capi.DQPSK, capi.R1_2, 40.0, 0.0)
    dem, enc = capi.OfdmDemodulator(ctx, cfg), capi.LdpcDecoder(ctx, capi.R1_2)
    for ncw in (1, 27):
        fr = torch.randint(0, 256, (n_frames, 40 + (ncw - 1) * 38), dtype=torch.uint8, device="cuda")
        w, got = dem.frame_tx_batch(enc, fr)
        assert got == ncw
        row = {}
        for rep in range(2):                                     # off, on, off, on: two rounds on the same inputs
            for bps in (0, dem.bits_per_symbol):
                dem.set_tx_interleave(bps)
                ms = timed(torch, lambda: dem.frame_tx_batch(enc, fr, out=w))
                row.setdefault("on" if bps else "off", []).append(round(ms, 3))
        dem.set_tx_interleave(0)
        out[f"ofdm_frame_tx_{ncw}cw"] = dict(frames=n_frames, ms_per_call=row)
        print("ofdm tx", ncw, row, flush=True)
    mc = capi.mcdpsk_config(8, 2)
    mdem = capi.McDpskDemodulator(ctx, mc)
    pay = torch.randint(0, 256, (n_frames, 40), dtype=torch.uint8, device="cuda")
    w = mdem.tx_batch(enc, pay)
    row = {}
    for rep in range(2):
        for bps in (0, 16):
            mdem.set_tx_interleave(bps)
            ms = timed(torch, lambda: mdem.tx_batch(enc, pay, out=w))
            row.setdefault("on" if bps else "off", []).append(round(ms, 3))
    out["mcdpsk_tx"] = dict(frames=n_frames, ms_per_call=row)
    print("mcdpsk tx", row, flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import torch
    from projectultra_b200 import build, capi
    build.build()
    ctx = capi.Context(0)
    res = dict(card=card(), deinterleave=bench_deinterleave(ctx, capi, torch), tx=bench_tx(ctx, capi, torch))
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(json.dumps(res) + "\n")


if __name__ == "__main__":
    main()
