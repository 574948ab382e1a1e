"""Quick demod-kernel-only timing of the bench workload (M1 512-FFT DQPSK presynced frames over AWGN), used during
development to compare kernel changes:
python tools/ofdm_quick_bench.py [frames_per_point] [mode: m1|m3]"""
import os
import sys

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
import numpy as np
import torch
from projectultra_b200 import capi, linksim

fpp = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
mode = sys.argv[2] if len(sys.argv) > 2 else "m1"
ctx = capi.Context(0)
if mode == "m1":
    cfg = capi.ModemConfig(48000, 1500, 512, 30, 1, 4, 2, 0, capi.DQPSK, capi.R1_2, 40.0, 0.0)
    snrs = [float(s) for s in range(-4, 9)]
    rate = capi.R1_2
elif mode == "m1qam16":       # M1 coherent, pilots/2 (tools/test_mode_snr.cpp:30)
    cfg = capi.ModemConfig(48000, 1500, 512, 30, 1, 4, 2, 1, capi.QAM16, capi.R1_2, 40.0, 0.0)
    snrs = [float(s) for s in range(4, 17)]
    rate = capi.R1_2
else:                          # M3: presets::nvis_mode() 1024-FFT 59 carriers CP 96, 32QAM R3/4 pilots/4 (config 3)
    cfg = capi.ModemConfig(48000, 1500, 1024, 59, 1, 0, 4, 1, capi.QAM32, capi.R3_4, 40.0, 0.0)
    snrs = [float(s) for s in range(6, 19)]
    rate = capi.R3_4
sim = linksim.LinkSim(ctx, cfg, os.environ.get("QB_CHANNEL", "awgn"), payload_bytes=40 if mode.startswith("m1") else 60, pool=64, code_rate=rate)
sim.ofdm.set_precision(os.environ.get("QB_PRECISION", "exact"))
n = len(snrs)
B = fpp * n
trials = np.repeat(np.arange(fpp, dtype=np.int64), n)
si = np.tile(np.arange(n, dtype=np.int64), fpp)
batch = sim.make_batch(snrs, si, trials)
rx = linksim.channel_apply(ctx, sim.ch, sim.tx_pool, batch["tx_index"], batch["noise_std"], batch["seed"])
llr = torch.zeros((B, 648), dtype=torch.float32, device="cuda")
for _ in range(3):
    sim.ofdm.presynced_batch(rx, 2, llr=llr, want_aux=False)
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
K = 10
e0.record()
for _ in range(K):
    sim.ofdm.presynced_batch(rx, 2, llr=llr, want_aux=False)
e1.record()
torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / K
alg = 4 * sim.L + 4 * 648
tag = " ".join("%s=%s" % (k, v) for k, v in sorted(os.environ.items()) if k.startswith("PU_"))
print("%-60s kernel=%s B=%d ms=%.4f  %.1f GB/s  %.1f Mframes/s  llr_crc=%08x" % (
    tag, sim.ofdm.last_kernel, B, ms, alg * B / ms / 1e6, B / ms / 1e3,
    int(llr.view(torch.int32).sum(dtype=torch.int64).item()) & 0xFFFFFFFF), flush=True)
