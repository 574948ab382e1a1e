"""LDPC decoder timing per case, for one or more builds of libpu_b200.so in one process.

    python tools/ldpc_quick_bench.py [--lib PATH ...] [--rounds N] [--min-ms MS] [--cases a,b,...]

Every --lib is loaded side by side (default: the in-tree build) and driven through its own C ABI on the same device
buffers, so two builds see identical inputs.  For every case the builds take turns, --rounds times, each turn timing
back-to-back launches with CUDA events over at least --min-ms of work.  One JSON line per (case, round, build).

Cases (LLRs as bench.py builds them):
  it0_53k, it0_1m, it1_53k, it1_1m   R1/2 at its waterfall (config 2), max_iter = 0 and 1: the per-codeword fixed cost
  headline                           the 53 248 LLR rows of bench.py's default run (M1 OFDM, 13 SNR points), max_iter = 50
  r12_easy, r12_waterfall, r12_stress, r14_easy, r14_waterfall, r14_stress
                                     config 2 (BPSK/AWGN, 1 M codewords) at R1/2 and R1/4, max_iter = 50
"""
import argparse
import ctypes as C
import json
import os
import sys

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from projectultra_b200 import capi  # noqa: E402

PU_MEM_DEVICE = 1
HEADLINE_B = 4096 * 13
K = {capi.R1_2: 324, capi.R1_4: 162}
SIGMA = {capi.R1_2: (0.5, 0.71, 0.95), capi.R1_4: (0.7, 1.12, 1.5)}   # easy / waterfall (bench.py --workload ldpc) / stress


class Build:
    """One libpu_b200.so: its own context and decoder handles."""

    def __init__(self, path):
        self.path = os.path.abspath(path)
        self.lib = L = C.CDLL(self.path)
        L.pu_status_string.restype = C.c_char_p
        L.pu_last_error.restype = C.c_char_p
        self.ctx = C.c_void_p()
        self.check(L.pu_init(0, C.byref(self.ctx)))
        self.decs = {}

    def check(self, st):
        if st != 0:
            raise RuntimeError("%s: %s: %s" % (self.path, self.lib.pu_status_string(st).decode(), self.lib.pu_last_error().decode()))

    def decoder(self, rate, max_iter):
        h = self.decs.get(rate)
        if h is None:
            h = self.decs[rate] = C.c_void_p()
            self.check(self.lib.pu_ldpc_create(self.ctx, rate, 50, C.byref(h)))
        self.check(self.lib.pu_ldpc_set_max_iterations(h, max_iter))
        return h

    def decode(self, h, llr, out):
        info, ok, it = out
        self.check(self.lib.pu_ldpc_decode_batch(h, C.c_void_p(llr.data_ptr()), C.c_size_t(llr.stride(0)), C.c_size_t(llr.shape[0]),
                                                 C.c_void_p(info.data_ptr()), C.c_size_t(info.stride(0)), C.c_void_p(ok.data_ptr()),
                                                 C.c_void_p(it.data_ptr()), PU_MEM_DEVICE,
                                                 C.c_void_p(torch.cuda.current_stream().cuda_stream)))


def config2_llr(rate, sigma, B, dev):
    """bench.py run_ldpc: 64 random codewords of the rate, BPSK over AWGN, LLR = clamp(2y/sigma^2, +-10)."""
    k = K[rate]
    rng = np.random.default_rng(100 + rate)
    cws = np.stack([np.unpackbits(capi.ldpc_encode(rate, rng.integers(0, 256, k // 8, dtype=np.uint8)))[:648] for _ in range(64)])
    bits = torch.from_numpy(cws.astype(np.float32)).to(dev)
    g = torch.Generator(device=dev)
    g.manual_seed(1)
    llr = torch.empty((B, 648), dtype=torch.float32, device=dev)
    for off in range(0, B, 1 << 18):
        n = min(1 << 18, B - off)
        y = (1 - 2 * bits)[(torch.arange(n, device=dev) + off) % 64] + sigma * torch.randn((n, 648), device=dev, generator=g)
        llr[off:off + n] = torch.clamp(2 * y / sigma ** 2, -10, 10)
    return llr


def headline_llr(dev):
    """The LLR rows bench.py's default run hands to the decoder (run_ours with --workload m1)."""
    import bench
    from projectultra_b200 import linksim
    wl = bench.WORKLOADS["m1"]
    c = list(wl["cfg"])
    c[8], c[9] = getattr(capi, c[8]), getattr(capi, c[9])
    ctx = capi.Context(0)
    sim = linksim.LinkSim(ctx, capi.ModemConfig(*c), wl["channel"], payload_bytes=wl["payload"], pool=bench.POOL,
                          code_rate=getattr(capi, wl["rate"]), precision="fast")
    fpp, n_snr = HEADLINE_B // len(wl["snr"]), len(wl["snr"])
    trials = np.repeat(np.arange(fpp, dtype=np.int64), n_snr)
    si = np.tile(np.arange(n_snr, dtype=np.int64), fpp)
    batch = sim.make_batch(wl["snr"], si, trials)
    rx = sim.make_rx(batch)
    B = fpp * n_snr
    bufs = dict(llr=torch.zeros((B, 648), dtype=torch.float32, device=dev),
                info=torch.empty((B, sim.ldpc.info_bytes), dtype=torch.uint8, device=dev),
                ok=torch.empty(B, dtype=torch.uint8, device=dev), iters=torch.empty(B, dtype=torch.int32, device=dev))
    sim.receive_count(batch, rx, torch.zeros((n_snr, 6), dtype=torch.int64, device=dev), bufs=bufs)
    torch.cuda.synchronize()
    return bufs["llr"]


def cases(dev):
    """(name, rate, max_iter, llr factory) in run order; the LLRs of a case exist only while it runs."""
    R12, R14 = capi.R1_2, capi.R1_4
    out = []
    for mi in (0, 1):
        out.append(("it%d_53k" % mi, R12, mi, lambda: config2_llr(R12, SIGMA[R12][1], HEADLINE_B, dev)))
        out.append(("it%d_1m" % mi, R12, mi, lambda: config2_llr(R12, SIGMA[R12][1], 1 << 20, dev)))
    out.append(("headline", R12, 50, lambda: headline_llr(dev)))
    for rate, tag in ((R12, "r12"), (R14, "r14")):
        for point, sigma in zip(("easy", "waterfall", "stress"), SIGMA[rate]):
            out.append(("%s_%s" % (tag, point), rate, 50, lambda rate=rate, sigma=sigma: config2_llr(rate, sigma, 1 << 20, dev)))
    return out


def time_case(b, h, llr, out, min_ms):
    """ms per launch over >= min_ms of back-to-back launches (after a warm-up launch that also sizes the window)."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    b.decode(h, llr, out)
    e1.record()
    torch.cuda.synchronize()
    n = max(3, int(min_ms / max(e0.elapsed_time(e1), 1e-3)) + 1)
    e0.record()
    for _ in range(n):
        b.decode(h, llr, out)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n, n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", action="append", help="libpu_b200.so to time (repeatable; default: the in-tree build)")
    ap.add_argument("--rounds", type=int, default=3, help="turns of every build per case")
    ap.add_argument("--min-ms", type=float, default=200.0, help="least GPU time per timed turn")
    ap.add_argument("--cases", help="comma-separated subset of the case names")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ldpc_quick_bench.py: no CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    builds = [Build(p) for p in (args.lib or [capi.LIB_PATH])]
    gpu = torch.cuda.get_device_name(0)
    want = set(args.cases.split(",")) if args.cases else None
    for name, rate, mi, make in cases(dev):
        if want and name not in want:
            continue
        llr = make()
        B = llr.shape[0]
        outs = [(torch.empty((B, (K[rate] + 7) // 8), dtype=torch.uint8, device=dev),
                 torch.empty(B, dtype=torch.uint8, device=dev), torch.empty(B, dtype=torch.int32, device=dev)) for _ in builds]
        for rnd in range(args.rounds):
            for b, out in zip(builds, outs):
                ms, n = time_case(b, b.decoder(rate, mi), llr, out, args.min_ms)
                info, ok, it = out
                print(json.dumps({"case": name, "lib": b.path, "round": rnd, "codewords": B, "rate": rate, "max_iter": mi,
                                  "ms": round(ms, 5), "launches": n, "ns_per_codeword": round(ms * 1e6 / B, 4),
                                  "iterations_run": float((it.float() + ok.float()).clamp(max=50).mean().item()),
                                  "converged": float(ok.float().mean().item()), "gpu": gpu}), flush=True)
        ref = outs[0]
        for b, out in zip(builds[1:], outs[1:]):   # every build decodes the same LLRs: outputs must agree
            same = all(bool(torch.equal(x, y)) for x, y in zip(ref, out))
            print(json.dumps({"case": name, "lib": b.path, "same_outputs_as": builds[0].path, "equal": same}), flush=True)
        del llr, outs
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
