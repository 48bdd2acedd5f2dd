"""Cost and quality of plan improvement by large-neighbourhood search on the device (`BatchedEnvironment.plan_lns`,
H = 256) against more priority orders (`plan_orders`), timed with CUDA events (median of 5 calls after 2 warm-up calls):
  - 8192 x 32 @ 40 and 4096 x 64 @ 80 from the device generator at density 0.3
  - the three golden test sets (tests/golden/instances_40_0.3.npz: 200 instances of 16 / 32 / 64 agents on 40 x 40)
For every batch: `plan()` and `plan_orders(R)` for R in {1, 4, 8, 16, 32}, then LNS with I in {1, 4, 16, 64} iterations x
neighbourhood k in {4, 8, 16} starting from `plan()` and from `plan_orders(R=8)`.  Each record has the call's time, the
solved fraction, the mean sum of costs over its solved environments, and the sum of costs over the environments every
method solves ("common"), so that LNS after plan_orders(8) (time: both calls) can be set against plan_orders(16 / 32) at
equal GPU time.  On the 16-agent set the project's CBS (`search.solve_batch`, node limit 2000 per instance) gives the gap
to the optimum on the instances both solve.  One JSON line per measurement to stdout and to --out (default
profiles/r3_pp_lns.jsonl); the card name and power limit are in every line.

    python profiles/tools/pp_lns_cost.py
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "..")
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from helpers import instances  # noqa: E402
from mapf_rl_b200 import BatchedEnvironment, search  # noqa: E402

H = 256
ORDERS = (1, 4, 8, 16, 32)
ITERATIONS = (1, 4, 16, 64)
NEIGHBOURHOODS = (4, 8, 16)
SEED = 0


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.strip().splitlines() or ["?, ?"])[0].split(", ")
    return name, power


def timed(fn, repeats=5, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(repeats):
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        out = fn()
        end.record()
        end.synchronize()
        ms.append(start.elapsed_time(end))
    return float(np.median(ms)), ms, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_pp_lns.jsonl"))
    ap.add_argument("--cbs-node-limit", type=int, default=2000)
    args = ap.parse_args()
    name, power = card()
    out = open(args.out, "w")

    def emit(rec):
        rec.update(horizon=H, seed=SEED, card=name, power_limit=power)
        line = json.dumps(rec)
        print(line, flush=True)
        out.write(line + "\n")
        out.flush()

    def sweep(env, shape, source, cbs=None):
        runs = {}
        med, ms, res = timed(lambda: env.plan(H))
        runs["plan"] = (med, ms, res, {})
        for R in ORDERS:
            med, ms, res = timed(lambda: env.plan_orders(H, R, SEED))
            runs[f"orders{R}"] = (med, ms, res, dict(orders=R))
        inputs = {"plan": runs["plan"], "plan_orders8": runs["orders8"]}
        for src, (in_ms, _, res, _) in inputs.items():
            for k in NEIGHBOURHOODS:
                for I in ITERATIONS:
                    med, ms, out_ = timed(lambda: env.plan_lns(res[0], res[1], I, k, SEED))
                    runs[f"lns_{src}_{I}_{k}"] = (med, ms, out_, dict(input=src, input_ms=in_ms, iterations=I, neighborhood=k))
        host = {key: tuple(x.cpu().numpy() for x in r[2]) for key, r in runs.items()}
        common = np.logical_and.reduce([h[2] >= 0 for h in host.values()])
        for key, (med, ms, _, extra) in runs.items():
            makespan, soc = host[key][2], host[key][3]
            ok = makespan >= 0
            rec = dict(what="pp_lns" if key.startswith("lns") else ("pp_plan" if key == "plan" else "pp_orders"), shape=shape,
                       source=source, ms=med, ms_all=ms, solved=float(ok.mean()),
                       soc_mean=float(soc[ok].mean()) if ok.any() else None, common=int(common.sum()),
                       soc_mean_common=float(soc[common].mean()) if common.any() else None, **extra)
            if key.startswith("lns"):
                acc = host[key][4]
                rec.update(total_ms=med + extra["input_ms"], accepted_mean=float(acc[acc >= 0].mean()) if (acc >= 0).any() else None)
            if cbs is not None:
                T, cost = cbs
                both = (T >= 0) & ok
                rec.update(cbs_node_limit=args.cbs_node_limit, cbs_solved=float((T >= 0).mean()), both=int(both.sum()),
                           cbs_soc_both=int(cost[both].sum()), soc_both=int(soc[both].sum()),
                           gap_to_cbs=float(soc[both].sum() / max(cost[both].sum(), 1) - 1.0))
            emit(rec)

    for B, N, L in ((8192, 32, 40), (4096, 64, 80)):
        env = BatchedEnvironment(B, N, L)
        env.reset(seed=1, env_offset=0, density=0.3)
        sweep(env, f"{B}x{N}@{L}", "generator density 0.3")
        env.close()
    for N in (16, 32, 64):
        maps, pos, goals = instances(N)
        env = BatchedEnvironment(len(maps), N, 40)
        env.load(maps, pos, goals)
        cbs = None
        if N == 16:
            dist = env.heuristic_distances().cpu().numpy()
            _, T, cost, _ = search.solve_batch(maps, pos, goals, dist=dist, time_limit_s=0, node_limit=args.cbs_node_limit)
            cbs = (T, cost)
        sweep(env, f"{len(maps)}x{N}@40", "tests/golden/instances_40_0.3.npz", cbs)
        env.close()
    out.close()


if __name__ == "__main__":
    main()
