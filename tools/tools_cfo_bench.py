"""Timing of the batched tools-CFO injector (pu_tools_cfo_apply_batch) and of the fresh-payload sweep on the chirp rows of the reduced table.

    python tools/tools_cfo_bench.py [--rows 4096] [--trials 16384] [--skip-sweep] [--out FILE.json]

Kernel time: CUDA events around 20 in-place calls on [rows, n] device rows (n = 68 812: OFDM_CHIRP + 480 + 2 400 samples of silence,
87 080: MC-DPSK behind the chirp + the same silence) after 3 warm-up calls; the 1.1-1.4 GB working set is larger than L2.  Sweep: the 13
chirp-acquired rows of `pu_sweep --table reduced` through pu_linksim_run on one GPU, pool vs fresh payloads.  The card's name and power
limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def chirp_rows(capi, fresh):
    """The chirp-acquired rows of tools/pu_sweep.cpp's reduced table (ofdm_mode / mcdpsk_mode with 480 + 2 400 samples of silence)."""
    m1 = capi.ModemConfig(48000, 1500, 512, 30, 1, 4, 2, 0, capi.DQPSK, capi.R1_2, 40.0, 0.0)
    m1r4 = capi.ModemConfig(48000, 1500, 512, 30, 1, 4, 2, 0, capi.DQPSK, capi.R1_4, 40.0, 0.0)
    mc = capi.mcdpsk_config(8, 2)
    kw = dict(peak=0.5, lead_samples=480, tail_samples=2400, fresh_payloads=fresh)
    t = [capi.sweep_mode(capi.WF_OFDM_CHIRP, m1, capi.R1_2, 40, "awgn", 5, 1, 16, precision="fast", cfo_hz=c, **kw) for c in (0.0, 30.0, 50.0)]
    t += [capi.sweep_mode(capi.WF_MCDPSK_CHIRP, mc, capi.R1_2, 40, ch, -6, 1, 22, cfo_hz=c, **kw)
          for ch in ("awgn", "moderate", "poor") for c in (0.0, 30.0, -30.0)]
    t += [capi.sweep_mode(capi.WF_OFDM_CHIRP, m1r4, capi.R1_4, 20, "moderate", 5, 1, 16, precision="fast", cfo_hz=30.0, **kw)]
    return t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=4096)
    ap.add_argument("--trials", type=int, default=16384)
    ap.add_argument("--skip-sweep", action="store_true")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import torch
    from projectultra_b200 import build, capi
    build.build()
    ctx = capi.Context(0)
    res = dict(card=card(), kernel={})
    for n in (68812, 87080):
        x = torch.randn((a.rows, n), dtype=torch.float32, device="cuda")
        h = capi.ToolsCfo(ctx, n, 30.0)
        for _ in range(3):
            h.apply_batch(x)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 20
        e0.record()
        for _ in range(reps):
            h.apply_batch(x)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        res["kernel"][str(n)] = dict(rows=a.rows, ms_per_call=round(ms, 3), us_per_row=round(1e3 * ms / a.rows, 3), rows_per_s=round(a.rows / ms * 1e3))
        print(n, res["kernel"][str(n)], flush=True)
        h.close()
        del x
    if not a.skip_sweep:
        res["chirp_rows"] = {}
        for fresh in (False, True):
            sw = capi.Sweep(chirp_rows(capi, fresh), trials_per_point=a.trials, block_trials=2048, pool=32)
            c, st = sw.run(ctx)
            res["chirp_rows"]["fresh" if fresh else "pool"] = dict(frames=int(st.frames_run), seconds=round(st.seconds, 3),
                                                                  setup_seconds=round(st.setup_seconds, 3), frames_per_s=round(st.frames_run / st.seconds),
                                                                  fer=(c[:, 1].astype(float) / c[:, 0]).round(4).tolist())
            print("fresh" if fresh else "pool", {k: v for k, v in res["chirp_rows"]["fresh" if fresh else "pool"].items() if k != "fer"}, flush=True)
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
