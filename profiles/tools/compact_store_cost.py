"""Cost of the compact replay store against the dense one, timed with CUDA events (medians over repeats; the two forms of
every operation are timed in turn inside each repeat):
  - step + observe into store rows, dense bytes vs packed bits: 8192 x 32 @ 40 uniform, 8192 x 6 @ 40 sized (reference level mix)
  - the comm mask alone and with packed rows written in the same launch
  - the actor's current frames: dense index_select vs mapf_obs_unpack (u8, and fp16)
  - the learner's window gather, dense vs compact, 192 samples x 18 frames x 32 agents
  - BatchedActor.step at C5's shape (2048 x 32 @ 40, 64-step episodes, bf16 Q-network), dense vs compact store
  - ReplayStore.nbytes at 16384 slots x 256 steps x 32 agents, and the largest power-of-two slot count of each layout that
    allocates next to an actor of 8192 environments x 32 agents (two actor steps run on it)
One JSON line per measurement to stdout and, with --out, to that file; the card name and power limit are in every line.

    python profiles/tools/compact_store_cost.py --out /tmp/r3_compact_store.jsonl
"""
import argparse
import gc
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", ".."))
from mapf_rl_b200 import BatchedEnvironment, ReplayStore  # noqa: E402
from mapf_rl_b200.actor import BatchedActor  # noqa: E402
from mapf_rl_b200.packed import unpack_obs  # noqa: E402
from mapf_rl_b200.qnet import Network  # noqa: E402

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


def compare(pairs, iters, repeats):
    """pairs: {name: fn}; warms every fn up, then times them in turn per repeat -> {name: [us]}"""
    for fn in pairs.values():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    t = {k: [] for k in pairs}
    for _ in range(repeats):
        for k, fn in pairs.items():
            t[k].append(time_us(fn, iters))
    return t


class AutocastNet:
    """the actor's Q-network forward under bf16 autocast, as profiles/bench_c5.py runs it"""

    def __init__(self, net):
        self.net = net

    def step(self, *a, **k):
        with torch.autocast("cuda", dtype=torch.bfloat16):
            return self.net.step(*a, **k)

    def reset(self):
        self.net.reset()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=8192)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--actor-envs", type=int, default=2048)
    ap.add_argument("--actor-steps", type=int, default=64)
    ap.add_argument("--skip-capacity", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    name, power = card()
    lines = []

    def emit(times, **kw):
        for k, v in times.items():
            lines.append(dict(kw, form=k, us_median=round(float(np.median(v)), 2), us_min=round(float(np.min(v)), 2),
                              us_max=round(float(np.max(v)), 2), repeats=len(v), gpu=name, power_limit=power))
        print(json.dumps(lines[-1]), flush=True)

    B = args.envs
    rng = np.random.default_rng(0)
    # ---- step + observe into store rows; comm mask; current-frame read ----
    for N, L, sized in ((32, 40, False), (6, 40, True)):
        env = BatchedEnvironment(B, N, L, device=dev, sized=sized)
        env.reset(seed=1, env_offset=0, density=0.3, levels=REF_LEVELS if sized else None)
        env.check()
        actions = torch.as_tensor(rng.integers(0, 5, size=(B, N)).astype(np.uint8), device=dev)
        rows = torch.arange(B, device=dev, dtype=torch.int64) * 2              # every other row, like a store's slots
        dense = torch.empty((2 * B, N, 6, 9, 9), dtype=torch.uint8, device=dev)
        bits = torch.empty((2 * B, N, 64), dtype=torch.uint8, device=dev)
        rewards = torch.empty((B, N), dtype=torch.float32, device=dev)
        done = torch.empty((B,), dtype=torch.uint8, device=dev)
        comm = torch.empty((B, N, N), dtype=torch.uint8, device=dev)
        cbits = torch.empty((2 * B, N, (N + 7) // 8), dtype=torch.uint8, device=dev)
        shape = dict(B=B, N=N, L=L, sized=sized)
        t = compare({"dense": lambda: env.step(actions, out_obs=dense, obs_rows=rows, out_rewards=rewards, out_done=done),
                     "packed": lambda: env.step(actions, out_bits=bits, obs_rows=rows, out_rewards=rewards, out_done=done)},
                    args.iters, args.repeats)
        emit(t, op="step_observe_rows", **shape)
        t = compare({"dense_only": lambda: env.comm_mask(out=comm),
                     "dense_and_packed_rows": lambda: env.comm_mask(out=comm, out_bits=cbits, rows=rows)}, args.iters, args.repeats)
        emit(t, op="comm_mask", **shape)
        t = compare({"dense_index_select_u8": lambda: dense.index_select(0, rows),
                     "unpack_u8": lambda: unpack_obs(bits, rows),
                     "unpack_f16": lambda: unpack_obs(bits, rows, dtype=torch.float16)}, args.iters, args.repeats)
        emit(t, op="current_frames", **shape)
        env.check()
        del env, dense, bits
        torch.cuda.empty_cache()

    # ---- learner window gather: 192 samples x 18 frames x 32 agents ----
    N, S, cap, batch = 32, 64, 1024, 192
    stores = {}
    for compact in (False, True):
        st = ReplayStore(cap, max_num_agents=N, device=dev, max_steps=S, compact=compact)
        for buf in ((st.obs_bits, st.comm_bits) if compact else (st.obs_buf, st.comm_mask)):
            buf.random_(0, 256 if compact else 2)
        st.hid_buf.normal_()
        st.size_buf.fill_(S)
        stores["compact" if compact else "dense"] = st
    slots = rng.integers(0, cap, size=batch)
    idx = torch.as_tensor(slots * S + rng.integers(0, S, size=batch), dtype=torch.int64, device=dev)
    t = compare({k: (lambda st=st: st.gather(idx)) for k, st in stores.items()}, args.iters, args.repeats)
    emit(t, op="gather", batch=batch, frames=18, N=N)
    del stores
    gc.collect()
    torch.cuda.empty_cache()

    # ---- actor step at C5's shape ----
    Ba, N, L, cap = args.actor_envs, 32, 40, 64
    slots = 1
    while slots < 2 * Ba:
        slots *= 2
    torch.manual_seed(0)
    net = Network().to(dev).to(memory_format=torch.channels_last).eval()
    actors = {}
    for compact in (False, True):
        env = BatchedEnvironment(Ba, N, L, device=dev)
        store = ReplayStore(slots, max_num_agents=N, device=dev, max_steps=cap, compact=compact)
        actors["compact" if compact else "dense"] = BatchedActor(env, AutocastNet(net), store, epsilon=0.2, seed=1, density=0.3,
                                                                  max_steps=cap)
    with torch.no_grad():
        t = compare({k: a.step for k, a in actors.items()}, args.actor_steps, args.repeats)
    emit(t, op="actor_step", B=Ba, N=N, L=L, max_steps=cap)
    for k, a in actors.items():
        a.env.check()
        lines.append(dict(op="actor_store_nbytes", form=k, B=Ba, slots=slots, max_steps=cap, nbytes=a.store.nbytes,
                          gpu=name, power_limit=power))
        print(json.dumps(lines[-1]), flush=True)
    del actors
    gc.collect()
    torch.cuda.empty_cache()

    # ---- capacity: 256-step episodes x 32 agents next to an actor of 8192 environments ----
    if not args.skip_capacity:
        N, L, S, Bc = 32, 40, 256, 8192
        for compact in (False, True):
            lines.append(dict(op="bytes_per_transition", form="compact" if compact else "dense", N=N, latent=256,
                              bytes=ReplayStore.bytes_per_transition(N, 256, compact), gpu=name, power_limit=power))
            print(json.dumps(lines[-1]), flush=True)
            largest, failures = None, []
            for cap in (1 << 18, 1 << 17, 1 << 16, 1 << 15, 1 << 14):
                env = store = actor = None
                try:
                    env = BatchedEnvironment(Bc, N, L, device=dev)
                    store = ReplayStore(cap, max_num_agents=N, device=dev, max_steps=S, compact=compact)
                    actor = BatchedActor(env, AutocastNet(net), store, epsilon=0.2, seed=1, density=0.3, max_steps=S)
                    with torch.no_grad():
                        actor.step()
                        actor.step()
                    torch.cuda.synchronize()
                    largest = dict(slots=cap, nbytes=store.nbytes, max_allocated=torch.cuda.max_memory_allocated())
                except RuntimeError as e:        # torch.OutOfMemoryError, or the sum tree's cudaMalloc (MapfError)
                    failures.append(dict(slots=cap, error=str(e).splitlines()[0][:160]))
                del env, store, actor
                gc.collect()
                torch.cuda.empty_cache()
                torch.cuda.reset_peak_memory_stats()
                if largest is not None:
                    break
            lines.append(dict(op="largest_slots_next_to_actor", form="compact" if compact else "dense", B=Bc, N=N, max_steps=S,
                              largest=largest, failed=failures, gpu=name, power_limit=power))
            print(json.dumps(lines[-1]), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(json.dumps(x) for x in lines) + "\n")


if __name__ == "__main__":
    main()
