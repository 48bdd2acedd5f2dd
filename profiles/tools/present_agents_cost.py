"""Cost of present-agent batches against padded ones, timed with CUDA events (medians of 5 repeats; the padded and the
present-only form are timed in turn inside each repeat):
  - BatchedActor.step at 8192 x 6 @ 40, sized, compact store, bf16 autocast on a channels_last network (as bench_c5 runs it),
    for three curriculum level sets: [(1, 10)], the first two growth rounds, the full 42 levels; with the observed per-step
    fill M / (B * N) of the present-only actor
  - the same actor at C5's uniform 2048 x 32 @ 40 (dense store, every agent present: the overhead of the index path)
  - a learner update (want_stats=False, 20 updates ending in a synchronise) from the store of the full-level actor
  - the two kernels against what they replace: unpack_obs + index_select, and the compact gather + the torch transpose / index
  - the encoder alone at batch sizes around the full-level fill: the first call of a new shape and the steady time per call
One JSON line per measurement to stdout and, with --out, to that file; the card name and power limit are in every line.

    python profiles/tools/present_agents_cost.py --out /tmp/r3_present_agents.jsonl
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", ".."))
from mapf_rl_b200 import BatchedEnvironment, ReplayStore, present  # noqa: E402
from mapf_rl_b200.actor import BatchedActor  # noqa: E402
from mapf_rl_b200.learner import BatchedLearner  # noqa: E402
from mapf_rl_b200.packed import unpack_obs  # noqa: E402
from mapf_rl_b200.qnet import Network  # noqa: E402

FULL = [(n, l) for n in range(1, 7) for l in range(10, 41, 5)]                  # 42 levels
TWO_ROUNDS = [(1, 10), (2, 10), (1, 15), (3, 10), (2, 15), (1, 20)]            # Curriculum defaults, two growth rounds
LEVEL_SETS = {"start": [(1, 10)], "two_rounds": TWO_ROUNDS, "full42": FULL}


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


def compare(pairs, iters, repeats=5, warm=3):
    for fn in pairs.values():
        for _ in range(warm):
            fn()
    torch.cuda.synchronize()
    t = {k: [] for k in pairs}
    for _ in range(repeats):
        for k, fn in pairs.items():
            t[k].append(time_us(fn, iters))
    return t


class AutocastNet:
    def __init__(self, net):
        self.net = net

    def step(self, *a, **k):
        with torch.autocast("cuda", dtype=torch.bfloat16):
            return self.net.step(*a, **k)

    def reset(self):
        self.net.reset()


def make_actor(net, B, N, L, cap, sized, compact, present_only, levels, seed=0):
    from mapf_rl_b200.curriculum import Curriculum
    env = BatchedEnvironment(B, N, L, device="cuda", sized=sized)
    cur = None
    if sized:
        cur = Curriculum(max_num_agents=N, max_map_length=L)
        for lv in levels:
            cur._add(lv)
    slots = 1
    while slots < 2 * B:
        slots *= 2
    store = ReplayStore(slots, max_num_agents=N, device="cuda", max_steps=cap, compact=compact)
    eps = 0.4 ** (1 + 7 * torch.arange(B, device="cuda", dtype=torch.float32) / max(B - 1, 1))
    return BatchedActor(env, AutocastNet(net), store, epsilon=eps, seed=seed, density=0.3, max_steps=cap, curriculum=cur,
                        present_only=present_only)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--steps", type=int, default=10, help="actor steps per timed repeat")
    ap.add_argument("--warm", type=int, default=160, help="actor warm-up steps (episode-length mix steady: 2.5 x the cap)")
    args = ap.parse_args()
    name, power = card()
    out = open(args.out, "w") if args.out else None

    def emit(**rec):
        rec.update(card=name, power_limit=power)
        line = json.dumps(rec)
        print(line, flush=True)
        if out:
            out.write(line + "\n")
            out.flush()

    torch.manual_seed(0)
    net = Network().cuda().eval().to(memory_format=torch.channels_last)
    cap = 64
    keep = {}

    # ---- actor step, sized 8192 x 6 @ 40 -------------------------------------------------------------------------------------
    B, N, L = 8192, 6, 40
    for tag, levels in LEVEL_SETS.items():
        actors = {m: make_actor(net, B, N, L, cap, True, True, m == "present", levels) for m in ("padded", "present")}
        for a in actors.values():
            a.run(args.warm)
        torch.cuda.synchronize()
        fills = []

        def step_present():
            actors["present"].step()
            fills.append(actors["present"].present.M / (B * N))

        t = compare({"padded": actors["padded"].step, "present": step_present}, args.steps, warm=1)
        emit(what="actor_step", shape=f"{B}x{N}@{L} sized compact bf16", levels=tag, n_levels=len(levels),
             padded_ms=float(np.median(t["padded"])) / 1e3, present_ms=float(np.median(t["present"])) / 1e3,
             padded_ms_all=[x / 1e3 for x in t["padded"]], present_ms_all=[x / 1e3 for x in t["present"]],
             fill_mean=float(np.mean(fills)), fill_min=float(np.min(fills)), fill_max=float(np.max(fills)),
             episodes=[actors["padded"].episodes, actors["present"].episodes])
        if tag == "full42":
            keep = actors
        else:
            del actors
        torch.cuda.empty_cache()

    # ---- learner update from the full-level stores ----------------------------------------------------------------------------
    learners = {m: BatchedLearner(net, keep[m].store, seed=1, present_only=m == "present") for m in ("padded", "present")}
    t = compare({m: (lambda l=l: l.update()) for m, l in learners.items()}, 20, warm=3)
    emit(what="learner_update", store=f"{B}x{N}@{L} full42 compact", batch=192,
         padded_ms=float(np.median(t["padded"])) / 1e3, present_ms=float(np.median(t["present"])) / 1e3,
         padded_ms_all=[x / 1e3 for x in t["padded"]], present_ms_all=[x / 1e3 for x in t["present"]],
         fill=learners["present"]._next[3]["present"].M / (192 * N))

    # ---- the kernels against what they replace ------------------------------------------------------------------------------
    a = keep["present"]
    st = a.store
    rows = a._rows()
    pr = a.present
    t = compare({"unpack+index_select": lambda: unpack_obs(st.obs_bits, rows).flatten(0, 1).index_select(0, pr.index),
                 "unpack_present": lambda: present.unpack_obs_present(st.obs_bits, rows, pr)}, 50)
    emit(what="current_frames_u8", shape=f"{B}x{N}", M=pr.M, M_pad=pr.M_pad,
         **{k + "_us": float(np.median(v)) for k, v in t.items()})
    idx = learners["present"]._next[0]
    counts = st.agents_buf[idx // st.max_steps]
    gpr = present.PresentRows(counts, int(counts.sum().item()), N)

    def padded_gather():
        o = st.gather(idx)
        W = st.bt_steps + st.forward_steps
        return gpr.select(o["obs"].transpose(1, 2).reshape(-1, W, 6, 9, 9)), gpr.select(o["hidden"])

    def present_gather():   # the kernel alone (the row count is read once, outside)
        import ctypes as C
        from mapf_rl_b200 import _native
        o = dict(obs=torch.empty((gpr.M_pad, 18, 6, 9, 9), dtype=torch.float16, device="cuda"),
                 comm_mask=torch.empty((192, 18, N, N), dtype=torch.uint8, device="cuda"),
                 hidden=torch.empty((gpr.M_pad, 256), dtype=torch.float16, device="cuda"))
        for k, dt in (("action", torch.int64), ("reward", torch.float16), ("done", torch.float16), ("steps", torch.float16),
                      ("bt_steps", torch.int64)):
            o[k] = torch.empty((192,), dtype=dt, device="cuda")
        batch = _native.ReplayBatch(*[o[k].data_ptr() for k in ("obs", "comm_mask", "hidden", "action", "reward", "done",
                                                                 "steps", "bt_steps")])
        _native.check(st._lib.mapf_replay_gather_present(C.byref(st._view()), C.c_void_p(st.agents_buf.data_ptr()),
                                                         C.c_void_p(idx.data_ptr()), C.c_void_p(gpr.first.data_ptr()), 192,
                                                         gpr.M_pad, C.byref(batch), None, st._stream()))
        return o

    t = compare({"compact_gather+transpose+index": padded_gather, "gather_present": present_gather,
                 "gather_present_with_M_read": lambda: st.gather(idx, present=True)}, 50)
    emit(what="window_gather", batch=192, W=18, N=N, M=gpr.M, M_pad=gpr.M_pad, **{k + "_us": float(np.median(v)) for k, v in t.items()})
    del learners, keep, a, st
    torch.cuda.empty_cache()

    # ---- encoder alone: first call of a new batch size and steady time, around the full-level fill ------------------------------
    enc = net.obs_encoder
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
        for M in (25600, 25601, 25856, 26112, 27000, 28672, 49152):
            x = torch.randint(0, 2, (M, 6, 9, 9), device="cuda").float().to(memory_format=torch.channels_last)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            enc(x)
            torch.cuda.synchronize()
            first_ms = (time.perf_counter() - t0) * 1e3
            steady = compare({"enc": lambda: enc(x)}, 10, warm=2)["enc"]
            emit(what="encoder_shape", M=M, first_call_ms=first_ms, steady_ms=float(np.median(steady)) / 1e3)

    # ---- actor step at C5's uniform shape: every agent present ----------------------------------------------------------------
    B, N, L = 2048, 32, 40
    actors = {m: make_actor(net, B, N, L, cap, False, False, m == "present", None) for m in ("padded", "present")}
    for a in actors.values():
        a.run(args.warm)
    t = compare({m: a.step for m, a in actors.items()}, args.steps, warm=1)
    emit(what="actor_step", shape=f"{B}x{N}@{L} uniform dense bf16 (C5)", levels="uniform",
         padded_ms=float(np.median(t["padded"])) / 1e3, present_ms=float(np.median(t["present"])) / 1e3,
         padded_ms_all=[x / 1e3 for x in t["padded"]], present_ms_all=[x / 1e3 for x in t["present"]], fill_mean=1.0)
    for a in actors.values():
        a.env.check()
    if out:
        out.close()


if __name__ == "__main__":
    main()
