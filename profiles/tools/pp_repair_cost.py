"""Cost and yield of plan repair by collision-based large-neighbourhood search on the device (`BatchedEnvironment.plan_repair`,
H = 256) against more priority orders (`plan_orders`), timed with CUDA events (median of 5 calls after 1 warm-up call):
  - 8192 x 32 @ 40 and 4096 x 64 @ 80 from the device generator at density 0.3
  - the three golden test sets (tests/golden/instances_40_0.3.npz: 200 instances of 16 / 32 / 64 agents on 40 x 40)
For every batch: `plan()`, `plan_orders(R)` for R in {8, 16, 32}, repair after `plan()` with I in {16, 64, 256} iterations x
neighbourhood k in {4, 8, 16}, repair after `plan_orders(8)` with the same I and k = 8, and repair of a batch with nothing
to repair (every arrival row 0: every environment passed through).  Each record has the call's time (and, for a repair, the
time with its input call), the solved fraction, the mean sum of costs over its solved environments and over the
environments every method solves ("common").  "Iterations used" by a repaired environment is the least I that repairs it
(the result does not depend on I once G = 0): on the golden sets it is found exactly by repairing with every I in 0 .. 64
(k = 8, after `plan()`); on the generated batches the records give the repaired count at each I.  One JSON line per
measurement to stdout and to --out (default profiles/r3_pp_repair.jsonl); the card name and power limit are in every line.

    python profiles/tools/pp_repair_cost.py
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
from mapf_rl_b200 import BatchedEnvironment  # noqa: E402

H = 256
ORDERS = (8, 16, 32)
ITERATIONS = (16, 64, 256)
NEIGHBOURHOODS = (4, 8, 16)
SEED = 0


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.strip().splitlines() or ["?, ?"])[0].split(", ")
    return name, power


def timed(fn, repeats=5, warm=1):
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
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_pp_repair.jsonl"))
    args = ap.parse_args()
    name, power = card()
    out = open(args.out, "w")

    def emit(rec):
        rec.update(horizon=H, seed=SEED, card=name, power_limit=power)
        line = json.dumps(rec)
        print(line, flush=True)
        out.write(line + "\n")
        out.flush()

    def sweep(env, shape, source, exact_iterations):
        runs = {}
        med, ms, res = timed(lambda: env.plan(H))
        runs["plan"] = (med, ms, res, {})
        for R in ORDERS:
            med, ms, res = timed(lambda: env.plan_orders(H, R, SEED))
            runs[f"orders{R}"] = (med, ms, res, dict(orders=R))
        grid = [("plan", I, k) for k in NEIGHBOURHOODS for I in ITERATIONS] + [("plan_orders8", I, 8) for I in ITERATIONS]
        for src, I, k in grid:
            in_ms, _, res, _ = runs["plan" if src == "plan" else "orders8"]
            med, ms, out_ = timed(lambda: env.plan_repair(res[0], res[1], I, k, SEED))
            runs[f"repair_{src}_{I}_{k}"] = (med, ms, out_, dict(input=src, input_ms=in_ms, iterations=I, neighborhood=k))
        host = {key: tuple(x.cpu().numpy() for x in r[2]) for key, r in runs.items()}
        common = np.logical_and.reduce([h[2] >= 0 for h in host.values()])
        for key, (med, ms, _, extra) in runs.items():
            makespan, soc = host[key][2], host[key][3]
            ok = makespan >= 0
            rec = dict(what="pp_repair" if key.startswith("repair") else ("pp_plan" if key == "plan" else "pp_orders"), shape=shape,
                       source=source, ms=med, ms_all=ms, solved=float(ok.mean()),
                       soc_mean=float(soc[ok].mean()) if ok.any() else None, common=int(common.sum()),
                       soc_mean_common=float(soc[common].mean()) if common.any() else None, **extra)
            if key.startswith("repair"):
                col = host[key][4]
                rec.update(total_ms=med + extra["input_ms"], input_failed=int((col != -2).sum()), repaired=int((col == 0).sum()),
                           unrepaired=int((col > 0).sum()), no_path=int((col == -1).sum()),
                           collisions_left_mean=float(col[col > 0].mean()) if (col > 0).any() else None)
            emit(rec)
        # pass-through: nothing to repair
        B, N = env.num_envs, env.num_agents
        zeros = (torch.zeros((H, B, N), dtype=torch.uint8, device="cuda"), torch.zeros((B, N), dtype=torch.int32, device="cuda"))
        med, ms, res = timed(lambda: env.plan_repair(zeros[0], zeros[1], 64, 8, SEED))
        emit(dict(what="pp_repair_pass_through", shape=shape, source=source, ms=med, ms_all=ms, iterations=64, neighborhood=8,
                  passed_through=int((res[4] == -2).sum().item())))
        if exact_iterations:
            base = runs["plan"][2]
            used = np.full(B, -1)
            for I in range(0, 65):
                col = env.plan_repair(base[0], base[1], I, 8, SEED)[4].cpu().numpy()
                used[(used < 0) & (col == 0)] = I
            rep = used >= 0
            failed = host["plan"][2] < 0
            emit(dict(what="pp_repair_iterations_used", shape=shape, source=source, input="plan", neighborhood=8, max_iterations=64,
                      input_failed=int(failed.sum()), repaired=int((rep & failed).sum()),
                      iterations_mean=float(used[rep & failed].mean()) if (rep & failed).any() else None,
                      iterations_median=float(np.median(used[rep & failed])) if (rep & failed).any() else None,
                      iterations_max=int(used[rep & failed].max()) if (rep & failed).any() else None,
                      initial_plan_collision_free=int((failed & (used == 0)).sum()),
                      within_3=int((rep & failed & (used <= 3)).sum())))

    for B, N, L in ((8192, 32, 40), (4096, 64, 80)):
        env = BatchedEnvironment(B, N, L)
        env.reset(seed=1, env_offset=0, density=0.3)
        sweep(env, f"{B}x{N}@{L}", "generator density 0.3", False)
        env.close()
    for N in (16, 32, 64):
        maps, pos, goals = instances(N)
        env = BatchedEnvironment(len(maps), N, 40)
        env.load(maps, pos, goals)
        sweep(env, f"{len(maps)}x{N}@40", "tests/golden/instances_40_0.3.npz", True)
        env.close()
    out.close()


if __name__ == "__main__":
    main()
