"""Cost of per-environment sizes: step + observe into replay-store rows, comm mask and level reset at B = 8192, timed with
CUDA events, for
  (a) a uniform (6, 40) handle,
  (b) a sized (6, 40) handle with every slot at (6, 40) -- the cost of the sized instantiations alone,
  (c) a sized (6, 40) handle drawing from the reference's full level set, n = 1..6 x l = 10, 15, ..., 40.
The three are timed in turn inside every repeat.  Writes one JSON line per (handle, operation) to stdout and, with
--out, to that file; the card name and power limit are part of every line.

    python profiles/tools/mixed_step_cost.py --out /tmp/mixed_step_cost.jsonl
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", ".."))
from mapf_rl_b200 import BatchedEnvironment  # noqa: E402

REF_LEVELS = [(n, l) for n in range(1, 7) for l in range(10, 41, 5)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.strip().splitlines() or ["?, ?"])[0].split(", ")
    return name, power


def time_us(fn, iters):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(iters):
        fn()
    end.record()
    end.synchronize()
    return start.elapsed_time(end) * 1000.0 / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=8192)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--reset-iters", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    B, N, L = args.envs, 6, 40
    dev = torch.device("cuda", 0)
    name, power = card()
    handles = {
        "a_uniform": (BatchedEnvironment(B, N, L, device=dev), None),
        "b_sized_full": (BatchedEnvironment(B, N, L, device=dev, sized=True), [(N, L)]),
        "c_sized_ref_levels": (BatchedEnvironment(B, N, L, device=dev, sized=True), REF_LEVELS),
    }
    rng = np.random.default_rng(0)
    actions = torch.as_tensor(rng.integers(0, 5, size=(B, N)).astype(np.uint8), device=dev)
    store = torch.empty((2 * B, N, 6, 9, 9), dtype=torch.uint8, device=dev)    # 48 MB: rows 2e, like a replay store
    rows = torch.arange(B, device=dev, dtype=torch.int64) * 2
    rewards = torch.empty((B, N), dtype=torch.float32, device=dev)
    done = torch.empty((B,), dtype=torch.uint8, device=dev)
    comm = torch.empty((B, N, N), dtype=torch.uint8, device=dev)
    ops = {}
    for key, (env, levels) in handles.items():
        env.reset(seed=1, env_offset=0, levels=levels)
        env.check()
        ops[key] = {
            "step_observe_rows": (lambda env=env: env.step(actions, out_obs=store, obs_rows=rows, out_rewards=rewards, out_done=done),
                                  args.iters),
            "comm_mask": (lambda env=env: env.comm_mask(out=comm), args.iters),
            "reset_levels": (lambda env=env, levels=levels: env.reset(seed=2, env_offset=B, levels=levels), args.reset_iters),
        }
        for fn, _ in ops[key].values():     # warm-up of every shape the timed window uses
            for _ in range(3):
                fn()
        env.check()
    torch.cuda.synchronize()
    times = {(k, o): [] for k in ops for o in ops[k]}
    for _ in range(args.repeats):
        for k in ops:
            for o, (fn, iters) in ops[k].items():
                times[(k, o)].append(time_us(fn, iters))
    for env, _ in handles.values():
        env.check()
    lines = []
    for (k, o), v in times.items():
        lines.append(dict(handle=k, op=o, B=B, N=N, L=L, us_median=round(float(np.median(v)), 2),
                          us_min=round(float(np.min(v)), 2), us_max=round(float(np.max(v)), 2), repeats=len(v),
                          gpu=name, power_limit=power))
    for k in ops:
        for o in ops[k]:
            base = np.median(times[("a_uniform", o)])
            lines.append(dict(handle=k, op=o, ratio_to_uniform=round(float(np.median(times[(k, o)]) / base), 4), gpu=name,
                              power_limit=power))
    text = "\n".join(json.dumps(x) for x in lines)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
