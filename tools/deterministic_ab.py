"""A/B of deterministic mode: alternate `bench.py` runs with CELLCOMM_B200_DETERMINISTIC unset
and =1, and record train cells/s at each of --batches (default: the benchmark's 2048 and the
reference's 128; one `bench.py --no-roofline --batch B` run each), with the card's name and
power limit read in the same run.

    python tools/deterministic_ab.py --reps 3 --out profiles/r03_deterministic_ab.json
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def bench(deterministic, batch, args):
    env = dict(os.environ)
    env.pop("CELLCOMM_B200_DETERMINISTIC", None)
    if deterministic:
        env["CELLCOMM_B200_DETERMINISTIC"] = "1"
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps",
           str(args.steps), "--warmup", str(args.warmup), "--batch", str(batch),
           "--small-batch", "0", "--no-cpu-baseline", "--no-roofline", "--dense-e2e-steps", "0"]
    r = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=1800)
    if r.returncode != 0:
        raise SystemExit(r.stderr[-3000:])
    # --no-roofline: bench.py prints the train numbers only ("value": resident-loop cells/s)
    line = json.loads([l for l in r.stdout.splitlines() if l.strip()][-1])
    assert line["metric"] == "BiGAN train cells/sec" and line["config"], line
    return line["value"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batches", type=int, nargs="+", default=[2048, 128])
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    gpu = card()
    runs = {f"batch_{b}": {"atomic": [], "deterministic": []} for b in args.batches}
    for _ in range(args.reps):
        for b in args.batches:
            runs[f"batch_{b}"]["atomic"].append(bench(False, b, args))
            runs[f"batch_{b}"]["deterministic"].append(bench(True, b, args))
    summary = {}
    for key, r in runs.items():
        a, d = statistics.median(r["atomic"]), statistics.median(r["deterministic"])
        summary[key] = {"atomic_cells_per_s": a, "deterministic_cells_per_s": d,
                        "deterministic_over_atomic": d / a}
    res = {"what": "bench.py train cells/s, CELLCOMM_B200_DETERMINISTIC unset vs =1, runs "
                   "alternated in one session; medians", "gpu (name, power limit, max SM clock)":
           gpu, "reps": args.reps, "steps": args.steps, "warmup": args.warmup,
           "median": summary, "runs": runs}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["median"]))


if __name__ == "__main__":
    main()
