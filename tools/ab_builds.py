#!/usr/bin/env python
"""A/B of two built trees of this repository on one GPU, alternating: base, new, base, new, ...

Each round runs, in each tree, `bench.py --no-e2e` (config 2, device-resident: value and CUDA-event time per stage)
and `bench_configs.py` (configs 3, 4 and 5s at reduced N: reads/s and stage times).  The first round also writes
`bench.py --dump-outputs` for both trees and compares the files byte for byte.  The card's name, power limit and SM
clocks are read before and after.  Every JSON line goes to <out>/ab.jsonl; a summary (min / median / max per tree)
is printed.

  python tools/ab_builds.py --base /path/to/parent/tree --new . --rounds 3 --out /tmp/ab
Both trees must be built (make -C biodemux.jl_b200/csrc) beforehand.
"""
from __future__ import annotations

import argparse
import filecmp
import json
import os
import statistics
import subprocess
import sys


def gpu_info():
    q = "name,power.limit,clocks.max.sm,clocks.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()[0]
        return dict(zip(q.split(","), [x.strip() for x in out.split(",")]))
    except Exception as e:  # reported, not fatal: the numbers are still worth having
        return {"error": str(e)}


def run_json(cmd, cwd):
    p = subprocess.run(cmd, cwd=cwd, capture_output=True, text=True)
    if p.returncode != 0:
        sys.stderr.write(p.stdout[-4000:] + p.stderr[-4000:])
        raise SystemExit(f"{' '.join(cmd)} in {cwd} failed with {p.returncode}")
    return [json.loads(ln) for ln in p.stdout.splitlines() if ln.startswith("{")]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base", required=True)
    ap.add_argument("--new", required=True)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--config-reads", type=int, default=2_000_000)
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    trees = {"base": os.path.abspath(args.base), "new": os.path.abspath(args.new)}
    log = open(os.path.join(args.out, "ab.jsonl"), "w")

    def emit(rec):
        log.write(json.dumps(rec) + "\n")
        log.flush()

    emit({"gpu_before": gpu_info()})
    rows = {k: [] for k in trees}
    cfg_rows = {k: [] for k in trees}
    for rnd in range(args.rounds):
        for name, tree in trees.items():
            cmd = [sys.executable, "bench.py", "--gpus", "1", "--steps", str(args.steps), "--warmup", "3", "--no-e2e"]
            if rnd == 0:
                cmd += ["--dump-outputs", os.path.join(os.path.abspath(args.out), f"dump_{name}")]
            (line,) = run_json(cmd, tree)
            rows[name].append(line)
            emit({"round": rnd, "tree": name, "bench": line})
            lines = run_json([sys.executable, "bench_configs.py", "--reads", str(args.config_reads), "--check", "2000",
                              "--steps", "5", "--only", "3", "4", "5s"], tree)
            cfg_rows[name].append(lines)
            for ln in lines:
                emit({"round": rnd, "tree": name, "config": ln})
    emit({"gpu_after": gpu_info()})

    da, db = (os.path.join(args.out, f"dump_{k}") for k in trees)
    files = sorted(os.listdir(da))
    same = files == sorted(os.listdir(db)) and all(filecmp.cmp(os.path.join(da, f), os.path.join(db, f), shallow=False)
                                                   for f in files)
    summary = {"dump_outputs_identical": same, "files": files}

    def mmm(xs):
        return [round(min(xs), 4), round(statistics.median(xs), 4), round(max(xs), 4)]

    for name in trees:
        r = rows[name]
        summary[name] = {"value_M": mmm([x["value"] / 1e6 for x in r]),
                         "ms_per_step": mmm([x["ms_per_step"] for x in r]),
                         "stage_ms_per_step": {k: mmm([x["stage_ms_per_step"].get(k, 0.0) for x in r])
                                               for k in r[0]["stage_ms_per_step"]},
                         "prefilter_fraction": mmm([x["prefilter_fraction"] for x in r])}
        per_cfg = {}
        for lines in cfg_rows[name]:
            for ln in lines:
                key = ln["config"].split(":")[0]
                per_cfg.setdefault(key, []).append(ln)
        summary[name]["configs"] = {k: {"reads_per_sec_M": mmm([x["reads_per_sec"] / 1e6 for x in v]),
                                        "k_prefilter_ms": mmm([x["stage_ms"].get("k_prefilter", 0.0) for x in v]),
                                        "reads_by_path": v[0]["reads_by_path"],
                                        "parity_bit_exact": all(x["parity_bit_exact"] for x in v)}
                                    for k, v in per_cfg.items()}
    emit({"summary": summary})
    print(json.dumps(summary, indent=1))


if __name__ == "__main__":
    main()
