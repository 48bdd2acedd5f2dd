"""Prioritized planning on the device (`BatchedEnvironment.plan`, mapf_env_plan_prioritized): exact parity with the numpy
restatement (tests/pp_ref.py) on generated batches, uniform and sized, plans that replay collision-free through the rollout
kernel and the oracle, properties against the BFS distances and the CBS expert, determinism, isolation between environments
and argument checks."""
import ctypes as C

import numpy as np
import pytest

import pp_ref
from cbs_cases import CBS_CASES, cbs_instance
from helpers import instances, random_instance
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


def _plan_np(env, H):
    out = env.plan(H)
    _torch().cuda.synchronize()
    return tuple(x.cpu().numpy() for x in out)


def _check_parity(plan, state, H, sample, n=None, l=None):
    actions, arrival, makespan, soc = plan
    maps, pos, goals = state
    for e in sample:
        ra, rr = pp_ref.plan(maps[e], pos[e], goals[e], H, None if n is None else n[e], None if l is None else l[e])
        assert np.array_equal(arrival[e], rr), (e, arrival[e].tolist(), rr.tolist())
        assert np.array_equal(actions[:, e], ra), e
        failed = (rr < 0).any()
        assert makespan[e] == (-1 if failed else rr.max()) and soc[e] == (-1 if failed else rr.sum()), e


def _sample(B, k, rng, must=()):
    return sorted(set(rng.choice(B, size=min(k, B), replace=False).tolist()) | set(int(e) for e in must))


def _check_rollout(env, plan, state, oracle_sample):
    """Replays the plan through the rollout kernel on `env` (loaded with the planned instances) and a few environments
    through the oracle: no collision before the episode ends, done first at step makespan - 1, everybody on the goal."""
    torch = _torch()
    actions, arrival, makespan, soc = plan
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
# 60 (3, 2), 80 (3, 3), 90 (4, 3), 120 (4, 4)
@pytest.mark.parametrize("B,N,L,k", [(300, 1, 6, 300), (257, 2, 7, 257), (600, 8, 12, 120), (128, 16, 30, 8), (512, 32, 40, 16),
                                     (64, 64, 40, 6), (64, 24, 60, 4), (32, 40, 80, 4), (32, 32, 90, 2), (16, 32, 120, 2)])
def test_parity_and_replay_generated(B, N, L, k):
    rng = np.random.default_rng(B * 1000 + N)
    env = _generated(B, N, L, seed=B + N + L)
    state = _state(env)
    plan = _plan_np(env, 256)
    assert (plan[2] >= 0).mean() > 0.5
    _check_parity(plan, state, 256, _sample(B, k, rng, np.flatnonzero(plan[2] < 0)[:4]))
    _check_rollout(env, plan, state, _sample(B, 3, rng))


@pytest.mark.parametrize("B,N,L,H", [(600, 8, 12, 8), (512, 32, 40, 64)])
def test_short_horizon_fails_some(B, N, L, H):
    rng = np.random.default_rng(H)
    env = _generated(B, N, L, seed=7 * H)
    state = _state(env)
    plan = _plan_np(env, H)
    failed = np.flatnonzero(plan[2] < 0)
    assert 0 < len(failed) < B
    for e in failed:
        assert (plan[1][e] == -1).all() and plan[3][e] == -1 and not plan[0][:, e].any()
    _check_parity(plan, state, H, _sample(B, 24, rng, failed[:8]))
    _check_rollout(env, plan, state, [])


def test_parity_sized_levels():
    from mapf_rl_b200 import BatchedEnvironment
    rng = np.random.default_rng(42)
    B = 1024
    env = BatchedEnvironment(B, 6, 40, sized=True)
    env.reset(seed=11, env_offset=0, density=0.3, levels=LEVELS)
    n, l = (x.cpu().numpy().astype(np.int64) for x in env.sizes)
    assert len(set(zip(n.tolist(), l.tolist()))) == len(LEVELS)
    state = _state(env)
    for H in (256, 12):
        plan = _plan_np(env, H)
        actions, arrival = plan[0], plan[1]
        ok = plan[2] >= 0
        assert ok.any()
        for e in np.flatnonzero(ok):
            assert (arrival[e, n[e]:] == 0).all() and not actions[:, e, n[e]:].any()
        # one environment of every level, and some more
        per_level = [int(np.flatnonzero((n == a) & (l == b))[0]) for a, b in LEVELS]
        _check_parity(plan, state, H, sorted(set(per_level) | set(_sample(B, 40, rng))), n=n, l=l)


def test_single_agent_arrival_is_bfs_distance():
    from mapf_rl_b200 import BatchedEnvironment
    from mapf_rl_b200.search import DIST_UNREACHABLE
    rng = np.random.default_rng(3)
    B, L, H = 300, 12, 12
    inst = [random_instance(rng, L, 1, 0.35) for _ in range(B)]
    maps, pos, goals = (np.stack(x) for x in zip(*inst))
    env = BatchedEnvironment(B, 1, L)
    env.load(maps, pos, goals)
    dist = env.heuristic_distances().cpu().numpy()
    _, arrival, makespan, soc = _plan_np(env, H)
    d = dist[np.arange(B), 0, pos[:, 0, 0], pos[:, 0, 1]]
    want = np.where((d == DIST_UNREACHABLE) | (d > H), -1, d)
    assert (d == DIST_UNREACHABLE).any() and ((d > H) & (d != DIST_UNREACHABLE)).any() and (want >= 0).any()
    assert np.array_equal(arrival[:, 0], want) and np.array_equal(makespan, want) and np.array_equal(soc, want)


def _cbs_bounds(maps, pos, goals, N, L, node_limit):
    from mapf_rl_b200 import BatchedEnvironment, search
    B = len(maps)
    env = BatchedEnvironment(B, N, L)
    env.load(maps, pos, goals)
    dist = env.heuristic_distances().cpu().numpy()
    _, _, makespan, soc = _plan_np(env, 256)
    _, T, cost, _ = search.solve_batch(maps, pos, goals, dist=dist, time_limit_s=0, node_limit=node_limit)
    both = (makespan >= 0) & (T >= 0)
    longest = dist[np.arange(B)[:, None], np.arange(N)[None, :], pos[..., 0], pos[..., 1]].max(1)
    assert (soc[both] >= cost[both]).all()
    assert (makespan[makespan >= 0] >= longest[makespan >= 0]).all()
    return both.sum(), makespan


def test_against_cbs_cases():
    both = 0
    for k, (L, N, density) in enumerate(CBS_CASES):
        m, s, g = cbs_instance(k, L, N, density)
        b, _ = _cbs_bounds(m[None].astype(np.uint8), s[None].astype(np.uint8), g[None].astype(np.uint8), N, L, 1 << 16)
        both += int(b)
    assert both >= 8


def test_against_cbs_golden_16():
    maps, pos, goals = instances(16)
    both, makespan = _cbs_bounds(maps, pos, goals, 16, 40, 2000)
    assert both >= 20 and (makespan >= 0).mean() > 0.5


def test_corridor_index_order_fails():
    from mapf_rl_b200 import BatchedEnvironment, search
    m, s, g = pp_ref.corridor_instance()
    env = BatchedEnvironment(1, 2, 5)
    env.load(m[None], s[None], g[None])
    actions, arrival, makespan, soc = _plan_np(env, 64)
    assert (arrival == -1).all() and makespan[0] == -1 and soc[0] == -1 and not actions.any()
    assert search.solve(m, s, g, time_limit_s=0)[0] is not None   # the instance is solvable


def test_determinism_and_isolation():
    rng = np.random.default_rng(5)
    B = 512
    env = _generated(B, 32, 40, seed=99)
    maps, pos, goals = _state(env)
    p1, p2 = _plan_np(env, 256), _plan_np(env, 256)
    for x, y in zip(p1, p2):
        assert np.array_equal(x, y)
    perm = rng.permutation(B)
    env.load(maps[perm], pos[perm], goals[perm])
    p3 = _plan_np(env, 256)
    assert np.array_equal(p3[0], p1[0][:, perm]) and np.array_equal(p3[1], p1[1][perm])
    assert np.array_equal(p3[2], p1[2][perm]) and np.array_equal(p3[3], p1[3][perm])


def test_arguments_and_state_unchanged():
    from mapf_rl_b200 import _native
    torch = _torch()
    env = _generated(64, 8, 12, seed=1)
    before = (env.agents_pos.cpu(), env.steps.cpu(), env.navi_map.cpu())
    bytes0 = env.arena_bytes
    lib, h, st = env._lib, env._h, env._stream()
    act = torch.zeros((1025, 64, 8), dtype=torch.uint8, device="cuda")
    arr = torch.zeros((64, 8), dtype=torch.int32, device="cuda")
    pa, pr = C.c_void_p(act.data_ptr()), C.c_void_p(arr.data_ptr())
    for H, a, r in ((0, pa, pr), (1025, pa, pr), (16, None, pr), (16, pa, None)):
        assert lib.mapf_env_plan_prioritized(h, H, a, r, st) == _native.MAPF_EINVAL
        assert b"mapf_env_plan_prioritized" in lib.mapf_last_error()
    assert lib.mapf_env_plan_prioritized(h, 1024, pa, pr, st) == _native.MAPF_OK
    env.plan(1)
    env.plan()
    env.check()
    after = (env.agents_pos.cpu(), env.steps.cpu(), env.navi_map.cpu())
    for x, y in zip(before, after):
        assert torch.equal(x, y)
    assert env.arena_bytes > bytes0
