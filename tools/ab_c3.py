"""A/B of the C3 benchmark between library builds of the same ABI: runs `bench.py --steps 4 --warmup 3 --no-e2e
--core-only --dump-outputs` once per build and round, alternating the builds (A, B, A, B, ...), and compares the distance
matrices each build dumped against the first build's.

    python tools/ab_c3.py OUT_DIR NAME=LIB.so [NAME=LIB.so ...] [--rounds 2]

OUT_DIR/<name>_<round>.json holds each bench line; OUT_DIR/summary.json the card, its power limit, the value ratios per
round and the largest relative difference of each build's matrices against the first build's (the dumps themselves are
deleted after the comparison)."""
import argparse
import json
import os
import shutil
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("builds", nargs="+", help="NAME=path/to/libngsdist_b200.so")
    ap.add_argument("--rounds", type=int, default=2)
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    builds = [b.split("=", 1) for b in args.builds]
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    lines = {name: [] for name, _ in builds}
    for rnd in range(args.rounds):
        for name, lib in builds:
            dump = os.path.join(args.out, "%s_%d" % (name, rnd))
            env = dict(os.environ, NGSDIST_B200_LIB=os.path.abspath(lib))
            cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "4", "--warmup", "3", "--no-e2e",
                   "--core-only", "--no-cpu-baseline", "--dump-outputs", dump]
            p = subprocess.run(cmd, env=env, capture_output=True, text=True, cwd=ROOT)
            if p.returncode:
                sys.stderr.write(p.stdout[-4000:] + p.stderr[-4000:])
                raise SystemExit("%s round %d failed" % (name, rnd))
            line = json.loads([ln for ln in p.stdout.splitlines() if ln.startswith("{")][-1])
            with open(dump + ".json", "w") as fh:
                json.dump(line, fh)
            lines[name].append(line)
            print("%s round %d: value %.4e  step %.1f ms  contraction %.1f ms  roofline.frac %.3f" % (
                name, rnd, line["value"], line["ms_per_step"], line["step_share_rank0_ms"]["contraction"], line["roofline"]["frac"]),
                flush=True)
    ref = builds[0][0]
    summary = {"card": card, "rounds": args.rounds, "builds": {}}
    for name, _ in builds:
        diffs = []
        for rnd in range(args.rounds):
            a = np.load(os.path.join(args.out, "%s_%d" % (ref, rnd), "dist.npy"))
            b = np.load(os.path.join(args.out, "%s_%d" % (name, rnd), "dist.npy"))
            with np.errstate(divide="ignore", invalid="ignore"):
                rel = np.abs(b - a) / np.abs(a)
            rel[(a == b) | (np.isnan(a) & np.isnan(b))] = 0.0
            k = int(np.nanargmax(rel))
            diffs.append({"max_rel": float(np.nanmax(rel)), "at": np.unravel_index(k, a.shape), "ref": float(a.flat[k]), "got": float(b.flat[k]),
                          "nan_pattern_equal": bool(np.array_equal(np.isnan(a), np.isnan(b)))})
        ls = lines[name]
        summary["builds"][name] = {
            "value": [x["value"] for x in ls],
            "value_ratio_vs_%s" % ref: [x["value"] / y["value"] for x, y in zip(ls, lines[ref])],
            "contraction_ms": [x["step_share_rank0_ms"]["contraction"] for x in ls],
            "contraction_ratio_vs_%s" % ref: [x["step_share_rank0_ms"]["contraction"] / y["step_share_rank0_ms"]["contraction"]
                                              for x, y in zip(ls, lines[ref])],
            "roofline_frac": [x["roofline"]["frac"] for x in ls],
            "dist_vs_%s" % ref: [{k: (list(map(int, v)) if k == "at" else v) for k, v in d.items()} for d in diffs],
        }
    for name, _ in builds:          # the matrices are compared above; only the JSON is kept
        for rnd in range(args.rounds):
            shutil.rmtree(os.path.join(args.out, "%s_%d" % (name, rnd)), ignore_errors=True)
    with open(os.path.join(args.out, "summary.json"), "w") as fh:
        json.dump(summary, fh, indent=1)
    print(json.dumps(summary, indent=1))


if __name__ == "__main__":
    main()
