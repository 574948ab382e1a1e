"""Timing of whole-frame FER: the batched multi-codeword transmitter (pu_frame_tx_batch) and the frame modes of the sweep driver.

    python tools/frame_sweep_bench.py [--frames 2048] [--trials 1024] [--out profiles/frame_sweep_bench.json]

Transmitter: CUDA events around 20 calls of pu_frame_tx_batch on [frames, frame_len] device rows (512-FFT DQPSK R1/2, layout 0, fresh
random frame bytes) after 3 warm-up calls, at 5, 40 and 255 codewords per frame; frames/s and output samples/s.  Sweep: every row of
`pu_sweep --table frames` (tools/pu_sweep.cpp) as a table of its own through pu_linksim_run on one GPU, pool vs fresh frames; frames/s and
codewords/s of the whole run (TX pool set-up excluded), and the transmitter's share of a fresh run = its event-timed time for the same
number of frames over the run time.  For the genie-timed rows the presynced kernel that serves them (pu_ofdm_last_kernel).  The card's
name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def frames_rows(capi, fresh, sizes=(200, 1000)):
    """The rows of tools/pu_sweep.cpp's frames table (ofdm_mode: chirp rows with 480 + 2 400 samples of silence and peak 0.5)."""
    m1 = lambda mod, pil: capi.ModemConfig(48000, 1500, 512, 30, 1, 4, 2, pil, mod, capi.R1_2, 40.0, 0.0)
    m3 = capi.ModemConfig(48000, 1500, 1024, 59, 1, 0, 4, 1, capi.QAM32, capi.R3_4, 40.0, 0.0)
    rows = []
    for size in sizes:
        for ch in ("awgn", "good", "poor"):
            step = 1.0 if ch == "awgn" else 2.0
            kw = dict(precision="fast", fresh_payloads=fresh, frame_payload_bytes=size)
            rows += [(f"512 DQPSK {size} B {ch}", capi.sweep_mode(capi.WF_OFDM, m1(capi.DQPSK, 0), capi.R1_2, 0, ch, -2, step, 12, **kw)),
                     (f"512 16QAM p/2 {size} B {ch}", capi.sweep_mode(capi.WF_OFDM, m1(capi.QAM16, 1), capi.R1_2, 0, ch, 6, step, 12, **kw)),
                     (f"1024 32QAM p/4 {size} B {ch}", capi.sweep_mode(capi.WF_OFDM, m3, capi.R3_4, 0, ch, 10, step, 12, **kw)),
                     (f"OFDM_CHIRP DQPSK {size} B {ch}", capi.sweep_mode(capi.WF_OFDM_CHIRP, m1(capi.DQPSK, 0), capi.R1_2, 0, ch, 0, step, 12, peak=0.5,
                                                                         lead_samples=480, tail_samples=2400, **kw))]
    return rows


def time_tx(ctx, capi, torch, n_frames, reps=20):
    cfg = capi.ModemConfig(48000, 1500, 512, 30, 1, 4, 2, 0, capi.DQPSK, capi.R1_2, 40.0, 0.0)
    dem, enc = capi.OfdmDemodulator(ctx, cfg), capi.LdpcDecoder(ctx, capi.R1_2)
    out = {}
    for ncw in (5, 40, 255):
        nbytes = 40 + (ncw - 1) * 38
        fr = torch.randint(0, 256, (n_frames, nbytes), dtype=torch.uint8, device="cuda")
        w, got = dem.frame_tx_batch(enc, fr)
        assert got == ncw
        for _ in range(3):
            dem.frame_tx_batch(enc, fr, out=w)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            dem.frame_tx_batch(enc, fr, out=w)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        out[str(ncw)] = dict(frames=n_frames, frame_len=int(w.shape[1]), ms_per_call=round(ms, 3), frames_per_s=round(n_frames / ms * 1e3),
                             samples_per_s=round(n_frames * w.shape[1] / ms * 1e3), us_per_frame=ms * 1e3 / n_frames)
        print("tx", ncw, out[str(ncw)], flush=True)
        del w, fr
    return out


def tx_us_per_frame(ctx, capi, torch, m, n_frames=1024, reps=10):
    """Event-timed pu_frame_tx_batch of one sweep row's frames (what a fresh batch runs per frame, before chirp, injector and noise)."""
    dem, enc = capi.OfdmDemodulator(ctx, m.ofdm), capi.LdpcDecoder(ctx, m.code_rate)
    fr = torch.randint(0, 256, (n_frames, m.frame_payload_bytes + 19), dtype=torch.uint8, device="cuda")
    w, _ = dem.frame_tx_batch(enc, fr, layout=1 if m.waveform == capi.WF_OFDM_SC else 0)
    dem.frame_tx_batch(enc, fr, out=w)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        dem.frame_tx_batch(enc, fr, out=w)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / reps / n_frames


def presynced_kernel(ctx, capi, m):
    dem, enc = capi.OfdmDemodulator(ctx, m.ofdm), capi.LdpcDecoder(ctx, m.code_rate)
    dem.set_precision("fast" if m.precision else "exact")
    import torch
    fr = torch.randint(0, 256, (4, m.frame_payload_bytes + 19), dtype=torch.uint8, device="cuda")
    w, ncw = dem.frame_tx_batch(enc, fr)
    dem.presynced_batch(w, 2, llr_stride=ncw * 648, want_aux=False)
    torch.cuda.synchronize()
    return dem.last_kernel


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=2048)
    ap.add_argument("--trials", type=int, default=1024)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import torch
    from projectultra_b200 import build, capi
    build.build()
    ctx = capi.Context(0)
    res = dict(card=card(), tx=time_tx(ctx, capi, torch, a.frames), sweep={})
    for (name, mp), (_, mf) in zip(frames_rows(capi, False), frames_rows(capi, True)):
        row = {}
        if mp.waveform == capi.WF_OFDM:
            row["presynced_kernel"] = presynced_kernel(ctx, capi, mp)
        for tag, m in (("pool", mp), ("fresh", mf)):
            sw = capi.Sweep([m], trials_per_point=a.trials, block_trials=1024, pool=32)
            c, st = sw.run(ctx)
            run_s = st.seconds - st.setup_seconds
            frames, cws = int(c[:, 0].sum()), int(c[:, 3].sum())
            row[tag] = dict(frames=frames, codewords_per_frame=cws // max(frames, 1), seconds=round(run_s, 3), setup_seconds=round(st.setup_seconds, 3),
                            frames_per_s=round(frames / run_s), codewords_per_s=round(cws / run_s),
                            fer=(c[:, 1].astype(float) / c[:, 0]).round(4).tolist())
        row["fresh"]["tx_share"] = round(tx_us_per_frame(ctx, capi, torch, mf) * 1e-6 * row["fresh"]["frames"] / row["fresh"]["seconds"], 4)
        res["sweep"][name] = row
        print(name, {t: {k: v for k, v in row[t].items() if k != "fer"} if isinstance(row[t], dict) else row[t] for t in row}, flush=True)
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
