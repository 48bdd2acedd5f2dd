"""Prioritized planning over several priority orders on the device (`BatchedEnvironment.plan_orders`,
mapf_env_plan_prioritized_orders): exact parity with the numpy restatement (tests/pp_orders_ref.py) on generated batches,
uniform and sized, bit-identity with `plan` at one order, monotonicity in the number of orders, plans that replay
collision-free through the rollout kernel and the oracle, sharding by env_offset, determinism and argument checks."""
import ctypes as C

import numpy as np
import pytest

import pp_orders_ref
import pp_ref
from helpers import instances
from oracle import oracle

pytestmark = pytest.mark.gpu

# the curriculum's settings as the sized-handle tests use them: 6 agent counts x 7 map sides
LEVELS = [(n, l) for n in range(1, 7) for l in range(10, 41, 5)]


def _torch():
    import torch
    return torch


def _generated(B, N, L, seed, density=0.3):
    from mapf_rl_b200 import BatchedEnvironment
    env = BatchedEnvironment(B, N, L)
    env.reset(seed=seed, env_offset=0, density=density)
    return env


def _state(env):
    return env.map.cpu().numpy(), env.agents_pos.cpu().numpy(), env.goals_pos.cpu().numpy()


def _plan_orders_np(env, H, R, seed=0, env_offset=0):
    out = env.plan_orders(H, R, seed, env_offset)
    _torch().cuda.synchronize()
    return tuple(x.cpu().numpy() for x in out)


def _plan_np(env, H):
    out = env.plan(H)
    _torch().cuda.synchronize()
    return tuple(x.cpu().numpy() for x in out)


def _check_parity(plan, state, H, R, seed, sample, n=None, l=None, env_offset=0):
    maps, pos, goals = state
    ref = pp_orders_ref.plan_orders_batch(maps, pos, goals, H, R, seed, env_offset, n, l, envs=sample)
    got = [x[:, sample] if i == 0 else x[sample] for i, x in enumerate(plan)]
    for name, x, y in zip(("actions", "arrival", "makespan", "soc", "order", "rank"), got, ref):
        assert np.array_equal(x, y), (name, [sample[i] for i in np.flatnonzero((x != y).reshape(len(sample), -1).any(1))]
                                      if name != "actions" else None)


def _sample(B, k, rng, must=()):
    return sorted(set(rng.choice(B, size=min(k, B), replace=False).tolist()) | set(int(e) for e in must))


def _check_rollout(env, plan, state, oracle_sample):
    """Replays the plan through the rollout kernel on `env` (loaded with the planned instances) and a few environments
    through the oracle: no collision before the episode ends, done first at step makespan - 1, everybody on the goal."""
    torch = _torch()
    actions, arrival, makespan = plan[:3]
    maps, pos, goals = state
    B, N = arrival.shape
    solved = makespan >= 0
    T = max(int(makespan.max()), 1)
    dev = torch.as_tensor(np.ascontiguousarray(actions[:T])).cuda()
    codes = torch.empty((T, B, N), dtype=torch.uint8, device="cuda")
    obs = torch.empty((1, B, N, 6, 9, 9), dtype=torch.uint8, device="cuda")
    _, _, done, _ = env.rollout(dev, num_steps=T, out_obs=obs, out_rewards=False, out_codes=codes)
    codes, done = codes.cpu().numpy(), done.cpu().numpy()
    final = env.agents_pos.cpu().numpy()
    for e in np.flatnonzero(solved):
        M = int(makespan[e])
        assert np.array_equal(final[e], goals[e]), e
        if M == 0:
            assert np.array_equal(pos[e], goals[e]), e
            continue
        assert not (codes[:M, e] == 3).any(), e
        assert not done[:M - 1, e].any() and done[M - 1, e] == 1, e
    for e in oracle_sample:
        if not solved[e]:
            continue
        o = oracle.OracleEnv()
        o.load(maps[e], pos[e], goals[e])
        M = int(makespan[e])
        for t in range(M):
            (_, p), rew, d, _ = o.step(np.asarray(actions[t, e], dtype=np.uint8))
            assert min(rew) > -0.5 + 1e-6 and bool(d) == (t == M - 1), (e, t)
        assert np.array_equal(np.asarray(o.agents_pos), goals[e])


# map sides 6 .. 120 cover every (row words, rows per lane) instance of the kernel: 6, 7, 12 (1, 1), 30 (2, 1), 40 (2, 2),
# 60 (3, 2), 80 (3, 3), 90 (4, 3), 120 (4, 4); k environments are compared at one order, fewer at more
@pytest.mark.parametrize("B,N,L,k", [(300, 1, 6, 60), (257, 2, 7, 60), (600, 8, 12, 40), (128, 16, 30, 8), (512, 32, 40, 8),
                                     (64, 64, 40, 4), (64, 24, 60, 4), (32, 40, 80, 2), (32, 32, 90, 2), (16, 32, 120, 2)])
def test_parity_generated(B, N, L, k):
    rng = np.random.default_rng(B * 1000 + N + 1)
    env = _generated(B, N, L, seed=B + N + L)
    state = _state(env)
    for R, seed in ((1, 0), (2, 5), (8, 77)):
        plan = _plan_orders_np(env, 256, R, seed)
        assert (plan[2] >= 0).mean() > 0.5
        failed = np.flatnonzero(plan[2] < 0)
        assert (plan[4][failed] == -1).all() and ((plan[4] >= 0) == (plan[2] >= 0)).all() and (plan[4] < R).all()
        sample = _sample(B, max(k // R, 1), rng)
        _check_parity(plan, state, 256, R, seed, sorted(set(sample) | set(failed[:2].tolist())))


def test_short_horizon_failures():
    rng = np.random.default_rng(8)
    B, N, L, H = 600, 8, 12, 8
    env = _generated(B, N, L, seed=7 * H)
    state = _state(env)
    plan = _plan_orders_np(env, H, 4, seed=3)
    failed = np.flatnonzero(plan[2] < 0)
    assert 0 < len(failed) < B
    for e in failed:
        assert (plan[1][e] == -1).all() and plan[3][e] == -1 and not plan[0][:, e].any()
        assert plan[4][e] == -1 and (plan[5][e] == 255).all()
    _check_parity(plan, state, H, 4, 3, _sample(B, 16, rng, failed[:8]))


def test_parity_sized_levels():
    from mapf_rl_b200 import BatchedEnvironment
    rng = np.random.default_rng(43)
    B = 1024
    env = BatchedEnvironment(B, 6, 40, sized=True)
    env.reset(seed=11, env_offset=0, density=0.3, levels=LEVELS)
    n, l = (x.cpu().numpy().astype(np.int64) for x in env.sizes)
    assert len(set(zip(n.tolist(), l.tolist()))) == len(LEVELS)
    state = _state(env)
    per_level = [int(np.flatnonzero((n == a) & (l == b))[0]) for a, b in LEVELS]
    for H in (256, 12):
        plan = _plan_orders_np(env, H, 8, seed=9)
        actions, arrival, makespan, _, order, rank = plan
        ok = makespan >= 0
        assert ok.any()
        for e in np.flatnonzero(ok):
            assert (arrival[e, n[e]:] == 0).all() and not actions[:, e, n[e]:].any() and (rank[e, n[e]:] == 255).all()
            assert sorted(rank[e, :n[e]].tolist()) == list(range(n[e]))
        # one environment of every level, and some more
        _check_parity(plan, state, H, 8, 9, sorted(set(per_level) | set(_sample(B, 24, rng))), n=n, l=l)
        # one order: plan()'s results
        one, base = _plan_orders_np(env, H, 1), _plan_np(env, H)
        for x, y in zip(one[:4], base):
            assert np.array_equal(x, y)


@pytest.mark.parametrize("B,N,L", [(600, 8, 12), (512, 32, 40), (64, 24, 60), (16, 32, 120)])
def test_one_order_is_plan(B, N, L):
    env = _generated(B, N, L, seed=3 * B + L)
    for H in (256, 24):
        base = _plan_np(env, H)
        one = _plan_orders_np(env, H, 1, seed=123, env_offset=9)
        for x, y in zip(one[:4], base):
            assert np.array_equal(x, y)
        solved = base[2] >= 0
        assert np.array_equal(one[4], np.where(solved, 0, -1))
        assert (one[5][solved] == np.arange(N, dtype=np.uint8)).all() and (one[5][~solved] == 255).all()


def _check_monotone(env, H):
    one = _plan_orders_np(env, H, 1)
    eight = _plan_orders_np(env, H, 8)
    s1, s8 = one[2] >= 0, eight[2] >= 0
    assert (s8 >= s1).all()
    assert (eight[3][s1] <= one[3][s1]).all()
    return one, eight


def test_monotone_in_orders_generated():
    env = _generated(2048, 32, 40, seed=21)
    one, eight = _check_monotone(env, 256)
    assert (eight[2] >= 0).sum() > (one[2] >= 0).sum()


def test_monotone_golden_64():
    from mapf_rl_b200 import BatchedEnvironment
    maps, pos, goals = instances(64)
    env = BatchedEnvironment(len(maps), 64, 40)
    env.load(maps, pos, goals)
    one, eight = _check_monotone(env, 256)
    assert (eight[2] >= 0).sum() > (one[2] >= 0).sum()
    # the restatement agrees on the first environments (tests/test_pp_orders_ref.py finds more solved there at 8 orders)
    k = 12
    _check_parity(eight, (maps, pos, goals), 256, 8, 0, list(range(k)))
    assert (eight[2][:k] >= 0).sum() > (one[2][:k] >= 0).sum()


def test_corridor_solved_by_another_order():
    from mapf_rl_b200 import BatchedEnvironment
    m, s, g = pp_ref.corridor_instance()
    seed = next(seed for seed in range(32) if pp_orders_ref.plan_orders(m, s, g, 64, 8, seed, 0)[2] >= 0)
    env = BatchedEnvironment(1, 2, 5)
    env.load(m[None], s[None], g[None])
    plan = _plan_orders_np(env, 64, 8, seed)
    assert plan[4][0] >= 1 and plan[5][0].tolist() == [1, 0] and plan[1][0].tolist() == [3, 4]
    _check_parity(plan, (m[None], s[None], g[None]), 64, 8, seed, [0])
    _check_rollout(env, plan, (m[None], s[None], g[None]), [0])


@pytest.mark.parametrize("B,N,L", [(512, 32, 40), (64, 24, 60)])
def test_replay(B, N, L):
    rng = np.random.default_rng(B + N)
    env = _generated(B, N, L, seed=5 * B + N)
    state = _state(env)
    plan = _plan_orders_np(env, 256, 8, seed=4)
    assert (plan[2] >= 0).mean() > 0.5
    _check_rollout(env, plan, state, _sample(B, 3, rng))


def test_sharding_and_determinism():
    from mapf_rl_b200 import BatchedEnvironment
    B, N, L, H, R, seed = 512, 32, 40, 256, 8, 31
    env = _generated(B, N, L, seed=17)
    maps, pos, goals = _state(env)
    whole = _plan_orders_np(env, H, R, seed)
    again = _plan_orders_np(env, H, R, seed)
    for x, y in zip(whole, again):
        assert np.array_equal(x, y)
    half = B // 2
    parts = []
    for off in (0, half):
        h = BatchedEnvironment(half, N, L)
        h.load(maps[off:off + half], pos[off:off + half], goals[off:off + half])
        parts.append(_plan_orders_np(h, H, R, seed, env_offset=off))
    for i, x in enumerate(whole):
        axis = 1 if i == 0 else 0
        assert np.array_equal(x, np.concatenate([p[i] for p in parts], axis=axis)), i
    # another seed draws other orders
    other = _plan_orders_np(env, H, R, seed + 1)
    assert not np.array_equal(other[5], whole[5])


def test_arguments_and_state_unchanged():
    from mapf_rl_b200 import _native
    torch = _torch()
    env = _generated(64, 8, 12, seed=1)
    before = (env.agents_pos.cpu(), env.steps.cpu(), env.navi_map.cpu())
    lib, h, st = env._lib, env._h, env._stream()
    act = torch.zeros((1025, 64, 8), dtype=torch.uint8, device="cuda")
    arr = torch.zeros((64, 8), dtype=torch.int32, device="cuda")
    order = torch.zeros(64, dtype=torch.int32, device="cuda")
    rank = torch.zeros((64, 8), dtype=torch.uint8, device="cuda")
    pa, pr, po, pk = (C.c_void_p(x.data_ptr()) for x in (act, arr, order, rank))
    for H, R, a, r, o, k in ((0, 4, pa, pr, po, pk), (1025, 4, pa, pr, po, pk), (16, 0, pa, pr, po, pk), (16, 257, pa, pr, po, pk),
                             (16, 4, None, pr, po, pk), (16, 4, pa, None, po, pk), (16, 4, pa, pr, None, pk),
                             (16, 4, pa, pr, po, None)):
        assert lib.mapf_env_plan_prioritized_orders(h, H, R, 0, 0, a, r, o, k, st) == _native.MAPF_EINVAL
        assert b"mapf_env_plan_prioritized_orders" in lib.mapf_last_error()
    assert lib.mapf_env_plan_prioritized_orders(h, 1024, 256, 0, 0, pa, pr, po, pk, st) == _native.MAPF_OK
    env.check()
    # the scratch: the planner tables of plan() plus one selection word per environment
    env2 = _generated(64, 8, 12, seed=1)
    bytes0 = env2.arena_bytes
    env2.plan(256)
    _torch().cuda.synchronize()
    bytes_plan = env2.arena_bytes
    assert bytes_plan > bytes0
    env3 = _generated(64, 8, 12, seed=1)
    env3.plan_orders(256, 1)
    _torch().cuda.synchronize()
    assert env3.arena_bytes == bytes_plan + 64 * 8
    env.plan_orders(1, 2)
    env.plan_orders()
    env.check()
    after = (env.agents_pos.cpu(), env.steps.cpu(), env.navi_map.cpu())
    for x, y in zip(before, after):
        assert torch.equal(x, y)
