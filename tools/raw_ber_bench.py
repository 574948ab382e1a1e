"""Cost of raw (pre-decoder) bit error counting in the sweep driver, and the raw table it produces.

    python tools/raw_ber_bench.py [--trials 8192] [--reps 3] [--out-dir profiles/raw_ber]

Runs `projectultra_b200/pu_sweep --table reduced` on one GPU without and with `--raw`, alternating (plain, raw, plain, raw, ...) so that a
drift of the shared machine hits both arms alike, `--reps` times each.  Per run it keeps the wall time of the process and the tool's own
summary (run-loop seconds, set-up / wait shares, launches); the rows of the last raw run go to raw_rows.jsonl.  The card's name, power
limit and maximum SM clock are read in the same call.  Writes <out-dir>/raw_ber_bench.json and <out-dir>/raw_rows.jsonl."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def run(exe, trials, raw, rows_path):
    cmd = [exe, "--table", "reduced", "--trials", str(trials), "--out", rows_path] + (["--raw"] if raw else [])
    env = dict(os.environ, RANK="0", WORLD_SIZE="1", LOCAL_RANK="0")
    t0 = time.perf_counter()
    r = subprocess.run(cmd, capture_output=True, text=True, env=env)
    wall = time.perf_counter() - t0
    if r.returncode != 0:
        sys.exit(f"{' '.join(cmd)} failed ({r.returncode}):\n{r.stderr[-4000:]}")
    with open(rows_path) as f:
        lines = [json.loads(x) for x in f if x.strip()]
    summary = [x for x in lines if x.get("summary")][-1]
    return dict(raw=raw, wall_seconds=round(wall, 3), summary=summary), [x for x in lines if not x.get("summary")]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--trials", type=int, default=8192)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out-dir", default=os.path.join(ROOT, "profiles", "raw_ber"))
    a = ap.parse_args()
    sys.path.insert(0, ROOT)
    from projectultra_b200 import build
    build.build()
    exe = os.path.join(ROOT, "projectultra_b200", "pu_sweep")
    os.makedirs(a.out_dir, exist_ok=True)
    tmp = os.path.join(a.out_dir, "rows.tmp.jsonl")
    runs, rows, plain_rows = [], None, None
    for i in range(a.reps):
        for raw in (False, True):
            res, r = run(exe, a.trials, raw, tmp)
            runs.append(res)
            print(json.dumps(res), flush=True)
            if raw:
                rows = r
            else:
                plain_rows = r
    os.remove(tmp)
    # the raw run's FER columns are those of the plain run: only the raw fields are added
    keys = [k for k in plain_rows[0] if k != "summary"]
    same = len(rows) == len(plain_rows) and all(all(x[k] == y[k] for k in keys) for x, y in zip(rows, plain_rows))
    sec = {raw: [r["summary"]["seconds"] for r in runs if r["raw"] == raw] for raw in (False, True)}
    out = dict(card=card(), trials_per_point=a.trials, table="reduced", runs=runs, plain_rows_equal_raw_rows_fer_columns=same,
               run_seconds_plain=sec[False], run_seconds_raw=sec[True],
               overhead_of_min=round(min(sec[True]) / min(sec[False]) - 1.0, 4))
    with open(os.path.join(a.out_dir, "raw_ber_bench.json"), "w") as f:
        json.dump(out, f, indent=1)
    with open(os.path.join(a.out_dir, "raw_rows.jsonl"), "w") as f:
        for r in rows:
            f.write(json.dumps(r) + "\n")
    print(json.dumps({k: v for k, v in out.items() if k != "runs"}))


if __name__ == "__main__":
    main()
