"""GPU: episode handling inside `rollout` at the sizes and in the sequence the benchmark runs it, with default tuning.

reset(seed, 0) -> set_autoreset(cap, seed, env_offset=B, stride=B) -> step counters staggered over [0, cap) -> a rollout
of 32 steps -> counters restaged -> a rollout of 20 steps into an observation ring of 4 and output rings of 2.  At these
sizes the library picks its own form of episode handling: re-generation inside the rollout kernel with the due slots
handed out first (C2 / C3), or staging by the dedicated generator / search kernels before the launch (C4); the second call
starts from flipped heuristic-map buffers and staged instances.  Everything is compared with a twin stepped launch by launch
whose finished slots are re-generated with reset(mask, env_offset + n * stride), and the re-generated instances of a sample
of slots with the host restatement of the generator (tests/generator_ref.py)."""
import numpy as np
import pytest

from generator_ref import generate
from oracle import oracle

pytestmark = pytest.mark.gpu

SEED, DENSITY, ACTION_SLOTS = 0, 0.3, 16
T1, T2, OBS_RING, OUT_RING = 32, 20, 4, 2


def greedy_script(env, T, seed):
    """Navi-greedy actions with epsilon 0.1 for T steps from the env's current state (each agent follows a set direction
    bit of its own cell, else stays); the env is restored afterwards."""
    import torch
    B, N = env.num_envs, env.num_agents
    g = torch.Generator(device=env.device)
    g.manual_seed(seed)
    pos0, steps0 = env.agents_pos.clone(), env.steps.clone()
    acts = torch.empty((T, B, N), dtype=torch.uint8, device=env.device)
    cur, _ = env.observe()
    for t in range(T):
        centre = cur[:, :, 2:6, 4, 4]
        pick = (centre.float() + torch.rand((B, N, 4), device=env.device, generator=g) * 0.5).argmax(-1) + 1
        greedy = torch.where(centre.any(-1), pick, torch.zeros_like(pick))
        eps = torch.rand((B, N), device=env.device, generator=g) < 0.1
        rnd = torch.randint(0, 5, (B, N), device=env.device, generator=g)
        acts[t] = torch.where(eps, rnd, greedy).to(torch.uint8)
        cur, _, _ = env.step(acts[t])
    env.set_state(agents_pos=pos0, steps=steps0)
    return acts


class Twin:
    """The episode handling of one rollout step through the public pieces: a slot that starts the step finished (all agents
    on their goals, or `cap` steps taken) gets instance n = (its episodes so far) + 1, reset(mask, env_offset + n * stride),
    and emits that instance's first observation with rewards 0, done 0, steps 0; every other slot steps."""

    def __init__(self, env, cap, env_offset, stride):
        self.env, self.cap, self.env_offset, self.stride = env, cap, env_offset, stride
        self.episode = np.zeros(env.num_envs, dtype=np.int64)

    def step(self, actions):
        import torch
        env = self.env
        fin = ((env.agents_pos == env.goals_pos).all(-1).all(-1) | (env.steps >= self.cap)).cpu().numpy()
        o, r, d = (x.clone() for x in env.step(actions))
        ids = np.flatnonzero(fin)
        for n in np.unique(self.episode[ids] + 1):
            mask = np.zeros(env.num_envs, dtype=np.uint8)
            mask[ids[self.episode[ids] + 1 == n]] = 1
            env.reset(mask=mask, seed=SEED, env_offset=self.env_offset + int(n) * self.stride, density=DENSITY)
        self.episode[ids] += 1
        if len(ids):
            m = torch.as_tensor(fin, device=env.device)
            o[m] = env.observe()[0][m]
            r[m] = 0
            d[m] = 0
        return o, r, d, env.steps.clone(), ids


def check_instances(events, B, L, N, what):
    """events: (slot, episode n, map, starts, goals, obs | None) of re-generated slots -> equal to the restated instance
    B + n * B + slot, and the observation emitted at the reset step equals the oracle's first observation of it."""
    for e, n, m, p, g, obs in events:
        rm, rp, rg, _ = generate(SEED, B + n * B + e, L, N, DENSITY)
        where = f"{what}: slot {e}, episode {n}"
        assert np.array_equal(m, rm), "map differs from the restated instance, " + where
        assert np.array_equal(p, rp) and np.array_equal(g, rg), "starts / goals differ from the restated instance, " + where
        if obs is not None:
            o = oracle.OracleEnv()
            o.load(rm, rp, rg)
            assert np.array_equal(obs, o.observe()[0].astype(np.uint8)), "first observation differs, " + where


@pytest.mark.parametrize("name,B,N,L,cap,actions", [("C2", 8192, 32, 40, 256, "uniform"),
                                                    ("C3", 8192, 64, 40, 256, "greedy"),
                                                    ("C4", 4096, 64, 80, 32, "uniform")])
def test_rollout_episode_handling_at_bench_scale(name, B, N, L, cap, actions):
    import torch
    from mapf_rl_b200 import BatchedEnvironment
    dev = torch.device("cuda", 0)
    env, twin_env = BatchedEnvironment(B, N, L, device=dev), BatchedEnvironment(B, N, L, device=dev)
    for e in (env, twin_env):
        e.reset(seed=SEED, env_offset=0, density=DENSITY)
    env.check()
    if actions == "greedy":
        acts = greedy_script(twin_env, ACTION_SLOTS, SEED)
    else:
        g = torch.Generator(device=dev)
        g.manual_seed(SEED)
        acts = torch.randint(0, 5, (ACTION_SLOTS, B, N), generator=g, device=dev, dtype=torch.uint8)
    env.set_autoreset(cap, seed=SEED, env_offset=B, stride=B, density=DENSITY)
    twin = Twin(twin_env, cap, B, B)
    stagger = ((torch.arange(B, device=dev, dtype=torch.int64) * 2654435761) % cap).to(torch.int32)
    # the slots sampled for the restatement: the ones whose cap falls inside the first call
    rng = np.random.default_rng(1)
    due = np.flatnonzero(stagger.cpu().numpy() + T1 > cap)
    sample = set(rng.choice(due, size=min(len(due), 64 if L <= 40 else 32), replace=False).tolist())
    events = []

    def record(ids, t, obs):
        picked = [e for e in ids if e in sample]
        if not picked:
            return
        idx = torch.as_tensor(picked, device=dev)
        m, p, g = (x[idx].cpu().numpy() for x in (twin_env.map, twin_env.agents_pos, twin_env.goals_pos))
        o = obs[t][idx].cpu().numpy() if obs is not None else [None] * len(picked)
        events.extend((e, int(twin.episode[e]), m[q], p[q], g[q], o[q]) for q, e in enumerate(picked))

    # ---- first call: full rings, every step against the twin ----
    for e in (env, twin_env):
        e.set_state(steps=stagger)
    obs, rew, done, steps = env.rollout(acts, num_steps=T1)
    env.check()                                    # nothing latched: generator, scheduler hand-over (MAPF_EINTERNAL)
    ep1 = env.episode_counts().cpu().numpy()
    resets1 = 0
    for t in range(T1):
        o, r, d, st, ids = twin.step(acts[t % ACTION_SLOTS])
        resets1 += len(ids)
        bad = (obs[t] != o).flatten(1).any(1).nonzero().flatten().tolist()
        assert not bad, (name, "call 1", t, bad[:8], len(bad))
        assert torch.equal(rew[t], r) and torch.equal(done[t], d) and torch.equal(steps[t], st), (name, "call 1", t)
        record(ids, t, obs)
    assert np.array_equal(ep1, twin.episode), (name, "episode counts after call 1")
    del obs, rew, done, steps

    # ---- second call: restaged counters, rings of 4 / 2 ----
    for e in (env, twin_env):
        e.set_state(steps=stagger)
    rings = [torch.zeros(sh, dtype=dt, device=dev) for sh, dt in
             (((OBS_RING, B, N, 6, 9, 9), torch.uint8), ((OUT_RING, B, N), torch.float32), ((OUT_RING, B), torch.uint8),
              ((OUT_RING, B), torch.int32))]
    env.rollout(acts, num_steps=T2, out_obs=rings[0], out_rewards=rings[1], out_done=rings[2], out_steps=rings[3])
    env.check()
    exp_obs, exp_out = {}, {}
    resets2 = 0
    for t in range(T2):
        o, r, d, st, ids = twin.step(acts[t % ACTION_SLOTS])
        resets2 += len(ids)
        if t >= T2 - OBS_RING:
            exp_obs[t % OBS_RING] = o
        if t >= T2 - OUT_RING:
            exp_out[t % OUT_RING] = (r, d, st)
        record(ids, t, None)
    for s in range(OBS_RING):
        bad = (rings[0][s] != exp_obs[s]).flatten(1).any(1).nonzero().flatten().tolist()
        assert not bad, (name, "call 2 obs ring", s, bad[:8], len(bad))
    for s in range(OUT_RING):
        r, d, st = exp_out[s]
        assert torch.equal(rings[1][s], r) and torch.equal(rings[2][s], d) and torch.equal(rings[3][s], st), (name, "call 2 ring", s)
    del rings, exp_obs

    # ---- final state, episode counts, re-generated instances ----
    assert torch.equal(env.agents_pos, twin_env.agents_pos) and torch.equal(env.goals_pos, twin_env.goals_pos), name
    assert torch.equal(env.map, twin_env.map) and torch.equal(env.steps, twin_env.steps), name
    assert torch.equal(env.navi_map, twin_env.navi_map), name
    counts = env.episode_counts().cpu().numpy()
    assert np.array_equal(counts, twin.episode), name
    assert resets1 > 0 and resets2 > 0 and int(counts.sum()) == resets1 + resets2
    assert int(counts.sum()) - int(ep1.sum()) == resets2
    assert len(events) >= len(sample)
    check_instances(events, B, L, N, name)
    last = sorted(e for e in sample if counts[e] > 0)
    idx = torch.as_tensor(last, device=dev)
    maps, goals = env.map[idx].cpu().numpy(), env.goals_pos[idx].cpu().numpy()
    for q, e in enumerate(last):
        rm, _, rg, _ = generate(SEED, B + int(counts[e]) * B + e, L, N, DENSITY)
        assert np.array_equal(maps[q], rm) and np.array_equal(goals[q], rg), (name, "final instance", e)
    env.check()
    twin_env.check()
    print(f"{name}: re-generations {resets1} in the {T1}-step call, {resets2} in the {T2}-step call; "
          f"{len(events)} checked against the restatement")
