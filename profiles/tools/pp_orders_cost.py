"""Cost and quality of prioritized planning over R priority orders on the device (`BatchedEnvironment.plan_orders`, H = 256)
for R in {1, 4, 8, 16, 32}, timed with CUDA events (median of 5 calls after 2 warm-up calls):
  - 8192 x 32 @ 40 and 4096 x 64 @ 80 from the device generator at density 0.3
  - the three golden test sets (tests/golden/instances_40_0.3.npz: 200 instances of 16 / 32 / 64 agents on 40 x 40)
with the solved fraction and the mean makespan / sum of costs over solved environments, `plan()` (index order) timed beside
each batch; and, on the 16-agent set, the CBS expert (`search.solve_batch`, the reference's 5-s limit per instance, all host
threads) against best-of-R: instances each solves that the other does not, and the sums of costs where both solve.
One JSON line per measurement to stdout and to --out (default profiles/r3_pp_orders.jsonl); the card name and power limit
are in every line.

    python profiles/tools/pp_orders_cost.py
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "..")
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from helpers import instances  # noqa: E402
from mapf_rl_b200 import BatchedEnvironment, search  # noqa: E402

H = 256
ORDERS = (1, 4, 8, 16, 32)
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
    return float(np.median(ms)), ms, tuple(x.cpu().numpy() for x in out)


def quality(makespan, soc):
    ok = makespan >= 0
    return dict(solved=float(ok.mean()), makespan_mean=float(makespan[ok].mean()) if ok.any() else None,
                soc_mean=float(soc[ok].mean()) if ok.any() else None)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_pp_orders.jsonl"))
    ap.add_argument("--cbs-time-limit", type=float, default=5.0, help="seconds per instance (the reference's limit)")
    args = ap.parse_args()
    name, power = card()
    out = open(args.out, "w")

    def emit(rec):
        rec.update(horizon=H, seed=SEED, card=name, power_limit=power)
        line = json.dumps(rec)
        print(line, flush=True)
        out.write(line + "\n")
        out.flush()

    def sweep(env, shape, source):
        res = {}
        med, ms, (_, _, makespan, soc) = timed(lambda: env.plan(H))
        emit(dict(what="pp_plan", shape=shape, source=source, ms=med, ms_all=ms, **quality(makespan, soc)))
        for R in ORDERS:
            before = env.arena_bytes
            med, ms, (_, _, makespan, soc, order, _) = timed(lambda: env.plan_orders(H, R, SEED))
            emit(dict(what="pp_orders", shape=shape, source=source, orders=R, ms=med, ms_all=ms,
                      scratch_grew_bytes=env.arena_bytes - before,
                      won_by_index_order=float((order == 0).mean()), **quality(makespan, soc)))
            res[R] = (makespan, soc)
        return res

    for B, N, L in ((8192, 32, 40), (4096, 64, 80)):
        env = BatchedEnvironment(B, N, L)
        env.reset(seed=1, env_offset=0, density=0.3)
        sweep(env, f"{B}x{N}@{L}", "generator density 0.3")
        env.close()
    for N in (16, 32, 64):
        maps, pos, goals = instances(N)
        env = BatchedEnvironment(len(maps), N, 40)
        env.load(maps, pos, goals)
        res = sweep(env, f"{len(maps)}x{N}@40", "tests/golden/instances_40_0.3.npz")
        if N == 16:
            dist = env.heuristic_distances().cpu().numpy()
            t0 = time.perf_counter()
            _, T, cost, _ = search.solve_batch(maps, pos, goals, dist=dist, time_limit_s=args.cbs_time_limit)
            wall = time.perf_counter() - t0
            cbs = T >= 0
            for R, (makespan, soc) in res.items():
                pp = makespan >= 0
                both = cbs & pp
                emit(dict(what="cbs_vs_pp_orders", shape=f"{len(maps)}x{N}@40", orders=R, cbs_wall_s=wall,
                          cbs_threads=os.cpu_count(), cbs_time_limit_s=args.cbs_time_limit, cbs_solved=float(cbs.mean()),
                          pp_solved=float(pp.mean()), both=int(both.sum()), cbs_soc_both=int(cost[both].sum()),
                          pp_soc_both=int(soc[both].sum()), pp_only=int((pp & ~cbs).sum()), cbs_only=int((cbs & ~pp).sum())))
        env.close()
    out.close()


if __name__ == "__main__":
    main()
