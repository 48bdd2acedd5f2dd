#!/usr/bin/env python
"""bench.py — env agent-steps/s of the fused step+observe hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config c2|c3|c4|c5] [--dump-outputs DIR]

One "step" = one lockstep Environment.step (+ the observe it ends in) over the whole batch of synthetic environments.
--config selects the BASELINE.json configuration (default c2 = configs[1], the one the metric is quoted on):
    c2  8192 envs x 32 agents, 40x40 / 0.3, uniform actions, episode cap 256 with reset inside the stepped path   (per GPU: weak)
    c3  8192 envs x 64 agents, 40x40 / 0.3, navi-greedy actions (congestion-heavy), sharded over the GPUs          (strong)
    c4  4096 envs x 64 agents, 80x80 / 0.3, episode cap 32: reset-heavy, exercises the BFS heuristic-map kernel    (per GPU: weak)
    c5  actor loop: 2048 envs x 32 agents + PyTorch Q-net forward + PER sum-tree / TD kernels + learner updates    (per GPU: weak)
Multi-GPU: env batches shard with no collective; torch.distributed is used only for the barrier and the max-over-ranks of
the device time (c5 adds the optional DDP all-reduce of the learner's gradients).

Printed JSON (rank 0, one line): see the field notes in DESIGN.md "Measurement".
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "env_agent_steps_per_sec_step_observe"
UNIT = "agent-steps/s"

CONFIGS = {
    "c2": dict(index=1, num_envs=8192, num_agents=32, map_length=40, density=0.3, actions="uniform", max_steps=256, scaling="weak"),
    "c3": dict(index=2, num_envs=8192, num_agents=64, map_length=40, density=0.3, actions="greedy", max_steps=256, scaling="strong"),
    "c4": dict(index=3, num_envs=4096, num_agents=64, map_length=80, density=0.3, actions="uniform", max_steps=32, scaling="weak"),
    "c5": dict(index=4, num_envs=2048, num_agents=32, map_length=40, density=0.3, actions="policy", max_steps=256, scaling="weak"),
}


def algo_bytes(N, L):
    """SURVEY.md 8(d): 486 obs + 40.5 navi crop + 1 action + 4 pos r/w + 2 goal + 4 reward + map/done/steps amortised."""
    return 486 + 40.5 + 1 + 4 + 2 + 4 + (L * L / 8.0 + 5) / N


def measured_hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def workload_name(args):
    c = CONFIGS[args.config]
    per = "per GPU" if args.scaling == "weak" else f"in total, sharded over {args.gpus} GPU(s)"
    extra = {"c2": "", "c3": ", navi-greedy actions (congestion-heavy)", "c4": ", reset-heavy (BFS heuristic maps)",
             "c5": " + PyTorch Q-net forward + PER sum-tree / TD kernels (actor loop)"}[args.config]
    return (f"batched step+observe, {args.map_length}x{args.map_length} / {args.density} density, {args.num_agents} agents, "
            f"{args.num_envs} lockstep envs {per}{extra} (BASELINE.json configs[{c['index']}])")


def make_instances(num, L, N, density, seed, first_index):
    """Synthetic batch following the reference generator (environment.py:100-138) at fixed density (host side)."""
    from concurrent.futures import ProcessPoolExecutor
    from mapf_rl_b200.instances import generate_batch
    workers = max(1, min(os.cpu_count() or 1, 32))
    chunk = (num + workers - 1) // workers
    jobs = [(min(chunk, num - s), L, N, density, seed, first_index + s) for s in range(0, num, chunk)]
    if workers == 1:
        parts = [generate_batch(*j) for j in jobs]
    else:
        with ProcessPoolExecutor(workers) as ex:
            parts = list(ex.map(generate_batch, *zip(*jobs)))
    return tuple(np.concatenate([p[i] for p in parts]) for i in range(3))


class ClockSampler:
    """Samples SM clock / throttle reasons of one GPU while the measured section runs (NVML, in-process)."""

    def __init__(self, index):
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _sample(self):
        nv = self.nv
        if nv is None:
            return
        try:
            self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
                     0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x100: "display_clock_setting"}
            for bit, name in names.items():
                if r & bit:
                    self.reasons.add(name)
        except Exception:
            pass

    def start(self):
        def run():
            while not self._stop.is_set():
                self._sample()
                time.sleep(0.001)
        self._t = threading.Thread(target=run, daemon=True)
        self._t.start()

    def stop(self):
        self._sample()
        self._stop.set()
        if self._t:
            self._t.join()
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s),
                "window": "the whole measured section: timed rollout, whole-batch launches, host-buffer steps (the K-step "
                          "rollout alone lasts under a millisecond)"}


# ---- CPU legs (the oracle port is the CHECKER; these are the only places bench.py executes it) ------------------------------
def port_setup(maps, agents, goals, threads):
    from oracle import oracle
    m = np.ascontiguousarray(np.asarray(maps) != 0, dtype=np.uint8)
    pos = np.ascontiguousarray(agents.astype(np.int32))
    gl = np.ascontiguousarray(goals.astype(np.int32))
    navi = oracle.navi_batch(m, gl, threads=threads)
    return m, pos, gl, navi


def port_run(state, acts, threads, bufs):
    """T lockstep steps of the C port over the batch, caller-owned output buffers (no allocation inside the timed loop)."""
    from oracle import oracle
    m, pos, gl, navi = state
    oracle.rollout(m, pos, gl, navi, acts, threads=threads, want_rewards=True, obs_out=bufs[0], done_out=bufs[1][:acts.shape[0]],
                   rewards_out=bufs[2][:acts.shape[0]])


def port_buffers(S, N, T):
    return (np.zeros((S, N, 6, 9, 9), dtype=np.uint8), np.zeros((T, S), dtype=np.uint8), np.zeros((T, S, N), dtype=np.float32))


def python_reference_leg(num_agents, seconds):
    """The reference's own Python Environment.step+observe, one process per core: timed live where the reference tree is
    mounted, else the committed result of the same script run in the dev container (the GPU box has no reference tree)."""
    try:
        from oracle import ref_loader, time_python_reference
        if ref_loader.available():
            r = time_python_reference.measure(num_agents if num_agents in (16, 32, 64) else 32, seconds)
            r["where"] = f"this box ({os.cpu_count()} host threads), live"
            return r
    except Exception as e:  # never let the optional leg break the bench line
        err = repr(e)
    else:
        err = None
    try:
        with open(os.path.join(ROOT, "profiles", "r2_python_reference_cpu.json")) as f:
            r = json.load(f)
        r["note"] = ("the reference tree is not present on this box: number measured by oracle/time_python_reference.py in the dev "
                     "container (core count in `cores`)" + (f"; live attempt failed: {err}" if err else ""))
        return r
    except Exception:
        return None


def cpu_baseline(maps, agents, goals, N, L, seconds=12.0, threads=None, max_envs=2048):
    """The oracle port (C restatement of environment.py:278-467) on the host cores, bounded sample."""
    threads = threads or (os.cpu_count() or 1)
    S = min(max_envs, maps.shape[0])
    state = port_setup(maps[:S], agents[:S], goals[:S], threads)
    rng = np.random.default_rng(1)
    T = 8
    acts = rng.integers(0, 5, size=(T, S, N)).astype(np.uint8)
    bufs = port_buffers(S, N, T)
    port_run(state, acts[:1], threads, bufs)  # warm
    t0 = time.perf_counter()
    done_steps = 0
    while True:
        port_run(state, acts, threads, bufs)
        done_steps += T
        el = time.perf_counter() - t0
        if el >= seconds:
            break
    out = {"value": S * N * done_steps / el, "unit": UNIT, "cores": threads, "kind": "port",
           "sample": f"{S} of the batch's envs x {done_steps} lockstep steps (uniform actions), C oracle port "
                     f"(oracle/mapf_oracle.c) on {threads} host threads, {el:.1f} s"}
    py = python_reference_leg(N, min(seconds, 8.0))
    if py:
        out["python_reference"] = py
    return out


def run_reference(args):
    """--impl reference: the reference's CPU algorithm for the path on this box's host cores (the C oracle port: the
    reference itself is pure Python and its tree does not exist on the GPU box), all host threads, rank 0 only, on the same
    config as the GPU arm: the whole batch of --num-envs environments per step, steps issued 8 per call into caller-owned
    buffers."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    N, L = args.num_agents, args.map_length
    threads = os.cpu_count() or 1
    S = args.num_envs if args.scaling == "weak" else args.num_envs   # one GPU's batch (weak) / the whole sharded batch (strong)
    maps, agents, goals = make_instances(S, L, N, args.density, args.seed, 0)
    state = port_setup(maps, agents, goals, threads)
    rng = np.random.default_rng(1)
    TC = 8
    acts = rng.integers(0, 5, size=(16, S, N)).astype(np.uint8)
    bufs = port_buffers(S, N, TC)

    def run(nsteps, start):
        s = start
        while nsteps > 0:
            t = min(TC, nsteps, 16 - s % 16)
            port_run(state, acts[s % 16:s % 16 + t], threads, bufs)
            nsteps -= t
            s += t
        return s

    pos = run(max(args.warmup, 1), 0)
    t0 = time.perf_counter()
    run(args.steps, pos)
    el = time.perf_counter() - t0
    value = S * N * args.steps / el
    sample = (f"each step = one lockstep step+observe over {S} envs ({N} agents, {L}x{L}, density {args.density}, uniform actions, "
              f"no episode resets: the port has no generator), C oracle port of environment.py:278-467 on {threads} host threads, "
              f"{TC} steps per call, caller-owned output buffers")
    cb = {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample}
    py = python_reference_leg(N, 6.0)
    if py:
        cb["python_reference"] = py
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * el / args.steps, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": bench_config(args),
            "method": {"timing": "time.perf_counter around the K steps on the host", "episodes": "no episode handling (the port has no generator)",
                       "instances": "host-side generator (mapf_rl_b200.instances), loaded into the port"},
            "cpu_baseline": cb,
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def bench_config(args, env=None, extra=None):
    """`config` of the JSON line: the workload, computed from the arguments alone, so that both arms (`--impl ours` and
    `--impl reference`) print the SAME object (the driver compares them); what is specific to an arm -- how it is timed, where
    its instances come from, its episode handling -- goes into the line's `method`."""
    world = max(1, args.gpus)
    per_gpu = args.num_envs // world if args.scaling == "strong" else args.num_envs
    obs_mb = per_gpu * args.num_agents * 486 / 1e6
    return {"workload": workload_name(args), "num_envs": args.num_envs, "num_agents": args.num_agents, "map_length": args.map_length,
            "obstacle_density": args.density, "actions": CONFIGS[args.config]["actions"], "config": args.config,
            "num_envs_per_gpu": per_gpu, "episode_cap": args.max_steps,
            "l2": (f"no flush: every step writes {obs_mb:.0f} MB of observations per GPU into the next slot of a rotating ring; the ring "
                   f"and the environments' state (heuristic maps) are several times the 126 MB L2")}


# ---- GPU arm -------------------------------------------------------------------------------------------------------------------
DUMP_BYTES = 48_000_000  # --dump-outputs writes at most this much


def last_step_sample(obs, rewards, done, steps):
    """--dump-outputs: what the rollout returned for its last step (observations uint8[B,N,6,9,9], rewards float32[B,N],
    done uint8[B], step counters int32[B]) as float32 host arrays, restricted to a fixed seeded sample of the environments
    so that the files stay under DUMP_BYTES; `env_index` names the sampled environments."""
    import torch
    B, N = rewards.shape
    per_env = 4 * (N * 6 * 9 * 9 + N + 2) + 8
    count = max(1, min(B, DUMP_BYTES // per_env))
    envs = np.sort(np.random.default_rng(0).choice(B, size=count, replace=False))
    idx = torch.as_tensor(envs, device=rewards.device)
    out = {name: t.index_select(0, idx).float().cpu().numpy()
           for name, t in (("obs", obs), ("rewards", rewards), ("done", done), ("steps", steps))}
    out["env_index"] = envs.astype(np.float64)
    return out


def write_dump(directory, arrays):
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def greedy_script(env, T, seed, device):
    """Navi-greedy actions with epsilon 0.1 (SURVEY 8(d) stream G) for T steps from the env's current state: each agent follows
    a set direction bit of its own cell (channels 2..5 of its observation), else stays.  The env is stepped while the script
    is recorded and restored afterwards (positions, step counters), so the timed rollout replays exactly these steps."""
    import torch
    B, N = env.num_envs, env.num_agents
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    pos0, steps0 = env.agents_pos.clone(), env.steps.clone()
    acts = torch.empty((T, B, N), dtype=torch.uint8, device=device)
    cur, _ = env.observe()
    for t in range(T):
        centre = cur[:, :, 2:6, 4, 4]
        pick = (centre.float() + torch.rand((B, N, 4), device=device, generator=g) * 0.5).argmax(-1) + 1
        greedy = torch.where(centre.any(-1), pick, torch.zeros_like(pick))
        eps = torch.rand((B, N), device=device, generator=g) < 0.1
        rnd = torch.randint(0, 5, (B, N), device=device, generator=g)
        acts[t] = torch.where(eps, rnd, greedy).to(torch.uint8)
        cur, _, _ = env.step(acts[t])
    env.set_state(agents_pos=pos0, steps=steps0)
    return acts


def run_ours(args):
    import torch
    import torch.distributed as dist
    from mapf_rl_b200 import BatchedEnvironment, sharding

    rank, world, local = sharding.rank_world()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    sharding.pin_to_cores(local, world)

    cfg = CONFIGS[args.config]
    N, L = args.num_agents, args.map_length
    if args.scaling == "strong":
        assert args.num_envs % world == 0, "strong scaling shards --num-envs evenly"
        B = args.num_envs // world
        first_env = rank * B
    else:
        B = args.num_envs
        first_env = sharding.weak_offset(B, rank)
    total_envs = B * world
    env = BatchedEnvironment(B, N, L, device=dev)
    # synthetic instances drawn on the device by the reference's procedure (environment.py:100-138) at fixed density; slot e of
    # rank r is global environment first_env + e whatever the number of GPUs
    env.reset(seed=args.seed, env_offset=first_env, density=args.density)
    env.check()

    K, A = args.steps, 16
    R = args.obs_ring  # observation ring (device replay slots): R x B*N*486 bytes > L2
    replay = torch.empty((R, B, N, 6, 9, 9), dtype=torch.uint8, device=dev)
    g = torch.Generator(device=dev)
    g.manual_seed(args.seed + rank)
    if cfg["actions"] == "greedy":
        A = max(16, min(K, 64))
        actions = greedy_script(env, A, args.seed + rank, dev)
    else:
        actions = torch.randint(0, 5, (A, B, N), generator=g, device=dev, dtype=torch.uint8)
    actions_host = actions[:16].cpu().pin_memory()  # page-locked: the host-buffer step hands slot s % 16 to the GPU in place
    actions_host = [actions_host[i] for i in range(actions_host.shape[0])]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # episode handling inside the stepped path (worker.py:390,422-428; SURVEY 8(d): cap 256, reset on done / cap).  The step
    # counters start staggered over [0, cap) -- the steady state of a pool of actors whose episodes end at different times --
    # so every rollout of K steps re-generates ~K / (cap + 1) of its environments (generator + BFS inside the launch).
    cap = 0 if args.no_autoreset else args.max_steps
    stagger = ((torch.arange(B, device=dev, dtype=torch.int64) * 2654435761) % max(cap, 1)).to(torch.int32)

    def arm(with_reset):
        if with_reset and cap > 0:
            env.set_autoreset(cap, seed=args.seed, env_offset=first_env + total_envs, stride=total_envs, density=args.density)
        else:
            env.set_autoreset(0)

    def restage():
        if cap > 0:
            env.set_state(steps=stagger)

    # warm-up: W whole-batch steps, then keep stepping until the clocks have had ~0.3 s of load
    arm(False)
    pos0, steps0 = env.agents_pos.clone(), env.steps.clone()
    for s in range(args.warmup):
        env.step(actions[s % A], out_obs=replay[s % R])
    t0 = time.perf_counter()
    s = 0
    while time.perf_counter() - t0 < 0.3:
        for _ in range(64):
            env.step(actions[s % A], out_obs=replay[s % R])
            s += 1
        torch.cuda.synchronize(dev)
    env.check()
    # the warm-up runs for a fixed time, so its number of steps varies: the timed region starts from the state before it, so
    # that the same arguments give the same inputs in every run
    env.set_state(agents_pos=pos0, steps=steps0)

    out_ring = 2
    rew_ring = torch.empty((out_ring, B, N), dtype=torch.float32, device=dev)
    done_ring = torch.empty((out_ring, B), dtype=torch.uint8, device=dev)
    steps_ring = torch.empty((out_ring, B), dtype=torch.int32, device=dev)

    def rollout(k):
        env.rollout(actions, num_steps=k, out_obs=replay, out_rewards=rew_ring, out_done=done_ring, out_steps=steps_ring,
                    chains=args.chains)

    def timed_rollout(k):
        """Device time of ONE mapf_env_rollout call of k steps.  The call is enqueued behind a short device-side spin, so the
        first event fires when the launch is already in the queue: the host's enqueue latency (~50 us of Python + driver, a
        tenth of a 20-step rollout) is not device time of the path."""
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        torch.cuda._sleep(args.gate_cycles)
        ev0.record()
        rollout(k)
        ev1.record()
        barrier()
        return ev0.elapsed_time(ev1)

    sampler = ClockSampler(local)
    chains, per, graph_period = env.rollout_plan(K, A, R, out_ring, args.chains)
    # ---- timed region: exactly K steps, device-resident inputs, episode resets inside ------------------------------------
    arm(True)
    restage()
    rollout(max(K, 32))        # untimed: first use of every code path (incl. a few re-generations)
    restage()
    torch.cuda.synchronize(dev)
    if cfg["actions"] == "greedy":
        pass                   # (the script was recorded from the state the env has been restored to; resets keep it "greedy-ish")
    sampler.start()
    ep0 = int(env.episode_counts().sum()) if cap > 0 else 0
    ms_local = timed_rollout(K)
    env.check()
    if args.dump_outputs and rank == 0:
        last = (K - 1) % R, (K - 1) % out_ring
        dump = last_step_sample(replay[last[0]], rew_ring[last[1]], done_ring[last[1]], steps_ring[last[1]])
    ms_all = sharding.gather_floats(ms_local, dev)
    ms = max(ms_all)
    value = world * B * N * K / (ms * 1e-3)
    resets_in_region = int(sharding.sum_over_ranks((int(env.episode_counts().sum()) - ep0) if cap > 0 else 0, dev))

    # ---- the same K steps without episode handling (what round 1 timed) --------------------------------------------------
    arm(False)
    restage()
    rollout(max(K, 32))
    ms_noreset = sharding.max_over_ranks(timed_rollout(K), dev)

    # ---- the same K steps as one whole-batch launch per step (mapf_env_step_observe from Python) ----
    ev2, ev3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev2.record()
    for s in range(K):
        env.step(actions[s % A], out_obs=replay[s % R])
    ev3.record()
    barrier()
    ms_single = sharding.max_over_ranks(ev2.elapsed_time(ev3), dev)

    # ---- e2e: through the host-buffer C-ABI entry point (mapf_env_step_host_codes) ---------------------
    replay_slots = [replay[i] for i in range(R)]

    def e2e_run(steps, codes=True):
        barrier()
        t0 = time.perf_counter()
        if codes:
            for s in range(steps):
                env.step_host_codes(actions_host[s % 16], device_obs=replay_slots[s % R])
        else:
            for s in range(steps):
                env.step_host(actions_host[s % 16], device_obs=replay_slots[s % R])
        torch.cuda.synchronize(dev)
        mine = time.perf_counter() - t0
        return mine

    e2e_steps = max(20, min(K, 400))
    e2e_run(32)   # warm-up
    # the host side of this path (Python, launch, flag poll) is sensitive to what else runs on the box: three
    # repetitions, the median is reported and all three are kept in the JSON line
    reps = []
    for _ in range(3):
        t_all = sharding.gather_floats(e2e_run(e2e_steps), dev)
        reps.append((world * B * N * e2e_steps / max(t_all), t_all))
    reps.sort(key=lambda x: x[0])
    e2e_value, e2e_times = reps[1]
    e2e_run(16, codes=False)
    t_f32 = sharding.max_over_ranks(e2e_run(max(10, min(K, 100)), codes=False), dev)
    e2e_f32_value = world * B * N * max(10, min(K, 100)) / t_f32
    clocks = sampler.stop()

    line = None
    if rank == 0:
        peak, peak_src = measured_hbm_peak()
        step_s = ms * 1e-3 / K
        ab = algo_bytes(N, L)
        achieved = ab * B * N / step_s / 1e9
        traffic = None
        try:
            with open(os.path.join(ROOT, "profiles", "rollout_traffic.json")) as f:
                traffic = json.load(f).get(args.config, {})
        except Exception:
            traffic = {}
        tr = traffic.get("dram_bytes_per_step")
        med = sorted(ms_all)[len(ms_all) // 2]
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": args.warmup,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": bench_config(args),
            "method": {
                "obs_ring_slots": R, "obs_ring_mb": round(R * B * N * 486 / 1e6), "state_arena_mb": round(env.arena_bytes / 1e6),
                "instances": "device-side generator (mapf_env_reset), global env index = first_env + slot",
                "episodes": (f"cap {cap} steps, reset on done / cap INSIDE the timed rollout (generator + BFS in the launch), step counters "
                             f"staggered over [0, {cap})" if cap > 0 else "no episode handling"),
                "extra_warmup": "0.3 s of untimed steps after W so SM clocks are under load",
                "timing": f"CUDA events on the launching stream around ONE mapf_env_rollout call of K steps, enqueued behind a "
                          f"{args.gate_cycles}-cycle device-side spin (host enqueue latency excluded); max over ranks"},
            "clocks": clocks,
            "gpu_launches": K * chains if chains else 1,
            "per_rank_ms": {"min": min(ms_all), "median": med, "max": max(ms_all), "all": ms_all},
            "launch": ({"api": "mapf_env_rollout (one call for the K steps)", "chains": chains, "envs_per_chain": per,
                        "graph_period_steps": graph_period}
                       if chains else
                       {"api": "mapf_env_rollout (one call for the K steps)", "chains": 0, "kernel": "rollout_kernel (persistent)",
                        "note": "ONE launch for the K steps: resident warps claim (environment, chunk of steps) work items time-major "
                                "from a global counter, keep the environment's state in registers / shared memory for the item, cache "
                                "each agent's 16x16 heuristic tile in shared memory, and re-generate finished environments in place"}),
            "episode_resets": {"cap": cap, "resets_in_timed_region": resets_in_region,
                               "ms_per_step_without_episode_handling": ms_noreset / K,
                               "value_without_episode_handling": world * B * N * K / (ms_noreset * 1e-3),
                               "cost_frac": (ms - ms_noreset) / ms_noreset},
            "single_launch": {"api": "mapf_env_step_observe, one whole-batch launch per step (no episode handling)",
                              "ms_per_step": ms_single / K, "value": world * B * N * K / (ms_single * 1e-3),
                              "roofline_frac": ab * B * N / (ms_single * 1e-3 / K) / 1e9 / peak},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": B * N, "d2h_bytes_per_step": B * N + B * 5,
                    "api": "mapf_env_step_host_codes on one of 16 page-locked action buffers, a two-stage pipeline: the step kernel reads "
                           "the actions in place over PCIe and ONE DMA copy brings u8 reward codes / steps / done back (internal stream); "
                           "the call returns when they are on the host, while the observe kernel writes the observation of a position "
                           "snapshot into the device replay ring on the caller's stream (north star), overlapping the next call's "
                           "step stage; timed with a device synchronize at the end",
                    "steps": e2e_steps, "repetitions": [r[0] for r in reps], "per_rank_s": e2e_times},
            "e2e_f32_rewards": {"value": e2e_f32_value, "unit": UNIT, "h2d_bytes_per_step": B * N, "d2h_bytes_per_step": B * N * 4 + B * 5,
                                "api": "mapf_env_step_host (fp32 rewards, step kernel -> observe kernel || D2H copies, CUDA graph, stream sync)"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": tr,
                         "frac_dram_bytes": (tr / step_s / 1e9 / peak) if tr else None,
                         "kernel": ("rollout_kernel<RW,K,2 warps> (persistent)" if not chains
                                    else "step_observe_kernel<RW,K,DO_STEP>"),
                         "per_launch": {"algorithmic_bytes": ab * B * N * (K if not chains else 1), "avg_duration_us": ms * 1e3 if not chains else step_s * 1e6,
                                        "steps_per_launch": K if not chains else 1},
                         "achieved_is": "algorithmic bytes of one whole-batch step / step period of the timed launch (its K steps "
                                        "overlap inside the launch); `traffic` = ncu dram__bytes_read+write of THIS kernel per step "
                                        "(profiles/rollout_traffic.json), frac_dram_bytes = traffic / step period / peak",
                         "traffic_source": traffic.get("source"),
                         "algorithmic_bytes_per_agent_step": ab, "peak_source": peak_src,
                         "note": "peak = measured copy (read+write) bandwidth; the rollout's traffic is almost write-only and a pure "
                                 "write stream reaches more than the copy figure on a B200, so frac can exceed 1"},
        }
        if not args.no_cpu_baseline and world == 1:
            S = min(2048, B)
            maps = env.map[:S].cpu().numpy()
            agents = env.agents_pos[:S].cpu().numpy()
            goals = env.goals_pos[:S].cpu().numpy()
            line["cpu_baseline"] = cpu_baseline(maps, agents, goals, N, L, seconds=args.cpu_seconds)
        print(json.dumps(line), flush=True)
        if args.dump_outputs:
            write_dump(args.dump_outputs, dump)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--num-envs", type=int, default=0)
    ap.add_argument("--num-agents", type=int, default=0)
    ap.add_argument("--map-length", type=int, default=0)
    ap.add_argument("--density", type=float, default=-1.0)
    ap.add_argument("--max-steps", type=int, default=0, help="episode cap (config default: 256; c4: 32)")
    ap.add_argument("--scaling", default="", choices=["", "weak", "strong"])
    ap.add_argument("--no-autoreset", action="store_true")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--obs-ring", type=int, default=4)
    ap.add_argument("--chains", type=int, default=0, help="sub-batch chains of mapf_env_rollout (0 = persistent kernel)")
    ap.add_argument("--gate-cycles", type=int, default=400_000)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--learner-every", type=int, default=4, help="c5: one learner update every this many actor steps")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write what the timed rollout returned for its last step (rank 0) as DIR/<name>.npy (c2, c3, c4)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    c = CONFIGS[args.config]
    args.num_envs = args.num_envs or c["num_envs"]
    args.num_agents = args.num_agents or c["num_agents"]
    args.map_length = args.map_length or c["map_length"]
    args.density = args.density if args.density >= 0 else c["density"]
    args.max_steps = args.max_steps or c["max_steps"]
    args.scaling = args.scaling or c["scaling"]
    if args.dump_outputs and (args.impl != "ours" or args.config == "c5"):
        ap.error("--dump-outputs is implemented for the rollout of --impl ours (configs c2, c3, c4)")

    if args.impl == "reference":
        run_reference(args)
        return
    if args.gpus > 1 and "WORLD_SIZE" not in os.environ:
        # launched by hand: re-exec under torchrun, one rank per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", str(29500 + os.getpid() % 1000), os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    if args.config == "c5":
        from profiles import bench_c5
        bench_c5.run(args, METRIC, UNIT, ClockSampler, measured_hbm_peak, workload_name, bench_config)
        return
    run_ours(args)


if __name__ == "__main__":
    main()
