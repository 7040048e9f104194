#!/usr/bin/env python
"""A/B of the allocate action's job order on the default bench workload (config3-cycle): keyed (default) vs replica
(KAI_JOB_ORDER=replica), in one process tree on one GPU so both arms see the same card and clocks.

  python profiles/r03_job_order_ab.py OUT_DIR [--runs 3] [--steps 20] [--warmup 5]

1. card name and power limit (nvidia-smi query, read only);
2. `bench.py --dump-outputs` once per arm: every array of the last step must be equal (visits included);
3. `bench.py --steps S --warmup W`, profiler off, alternating keyed / replica, `--runs` of each: ms_per_step per run;
4. one `KAI_PROFILE=1 bench.py --steps 2 --warmup 1` per arm for the host sequencer's rdtsc sections.
Writes OUT_DIR/summary.json and the raw logs; exits non-zero when the outputs differ."""
import argparse
import glob
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def bench(args, env_extra, log):
    env = dict(os.environ)
    env.pop("KAI_JOB_ORDER", None)
    env.pop("KAI_PROFILE", None)
    env.update(env_extra)
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1"] + args, env=env,
                       capture_output=True, text=True, cwd=ROOT)
    with open(log, "w") as f:
        f.write(p.stderr)
        f.write(p.stdout)
    if p.returncode != 0:
        raise SystemExit(f"bench.py {args} {env_extra} failed ({p.returncode}); see {log}")
    line = [x for x in p.stdout.splitlines() if x.startswith("{")][-1]
    return json.loads(line), p.stderr


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    arms = {"keyed": {}, "replica": {"KAI_JOB_ORDER": "replica"}}
    summary = {"gpu": subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                     capture_output=True, text=True).stdout.strip()}
    # same results
    dumps = {}
    for name, env in arms.items():
        d = os.path.join(a.out, f"dump_{name}")
        r, _ = bench(["--steps", "1", "--warmup", "1", "--dump-outputs", d], env, os.path.join(a.out, f"dump_{name}.log"))
        dumps[name] = d
        summary[f"dump_{name}"] = {k: r.get(k) for k in ("bindings_match", "victims_match", "node_tables_match")}
    files = sorted(os.path.basename(f) for f in glob.glob(os.path.join(dumps["keyed"], "*.npy")))
    other = sorted(os.path.basename(f) for f in glob.glob(os.path.join(dumps["replica"], "*.npy")))
    diff = [f for f in files if f not in other or not np.array_equal(np.load(os.path.join(dumps["keyed"], f)),
                                                                      np.load(os.path.join(dumps["replica"], f)))]
    summary["arrays_compared"] = len(files)
    summary["arrays_differing"] = diff + [f for f in other if f not in files]
    # speed, profiler off, alternating arms
    ms = {name: [] for name in arms}
    for i in range(a.runs):
        for name, env in arms.items():
            r, _ = bench(["--steps", str(a.steps), "--warmup", str(a.warmup)], env, os.path.join(a.out, f"run{i}_{name}.log"))
            ms[name].append(r["ms_per_step"])
            print(f"run {i} {name}: ms_per_step {r['ms_per_step']:.3f} e2e {r['e2e']['ms_per_step']:.3f}", flush=True)
    summary["ms_per_step"] = ms
    summary["spread_ms"] = {k: max(v) - min(v) for k, v in ms.items()}
    summary["min_replica_minus_max_keyed_ms"] = min(ms["replica"]) - max(ms["keyed"])
    # rdtsc sections, profiler on
    for name, env in arms.items():
        _, err = bench(["--steps", "2", "--warmup", "1"], dict(env, KAI_PROFILE="1"), os.path.join(a.out, f"profile_{name}.log"))
        summary[f"profile_{name}"] = [x for x in err.splitlines() if "rdtsc" in x or "job order" in x][-4:]
    with open(os.path.join(a.out, "summary.json"), "w") as f:
        json.dump(summary, f, indent=1)
    print(json.dumps(summary, indent=1))
    if summary["arrays_differing"] or not files:
        raise SystemExit("keyed and replica outputs differ")


if __name__ == "__main__":
    main()
