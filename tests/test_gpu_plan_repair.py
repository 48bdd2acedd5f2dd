"""Plan repair by collision-based large-neighbourhood search on the device (`BatchedEnvironment.plan_repair`,
mapf_env_plan_repair): exact parity with the numpy restatement (tests/pp_repair_ref.py) on generated batches, uniform and
sized, from plan() and plan_orders() output, with passed-through (-2), unplannable (-1), repaired (0) and unrepaired (> 0)
environments in the samples; plan()'s plan wherever plan() solves; repaired plans as plan_lns input and through the rollout
kernel and the oracle; determinism, sharding by env_offset, the handle's state and the caller's tensors unchanged; argument
checks and the scratch in mapf_env_arena_bytes; the 64-agent golden set and bounds against the project's CBS."""
import ctypes as C

import numpy as np
import pytest

import pp_repair_ref
from cbs_cases import CBS_CASES, cbs_instance
from helpers import instances
from test_gpu_plan_orders import LEVELS, _check_rollout

pytestmark = pytest.mark.gpu


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


def _np(out):
    _torch().cuda.synchronize()
    return tuple(x.cpu().numpy() for x in out)


def _repair_np(env, plan, I, k, seed=0, env_offset=0):
    return _np(env.plan_repair(plan[0], plan[1], I, k, seed, env_offset))


def _check_parity(got, state, inp, I, k, seed, sample, n=None, l=None, env_offset=0):
    maps, pos, goals = state
    ref = pp_repair_ref.plan_repair_batch(maps, pos, goals, inp[0], inp[1], I, k, seed, env_offset, n, l, envs=sample)
    mine = [x[:, sample] if i == 0 else x[sample] for i, x in enumerate(got)]
    for name, x, y in zip(("actions", "arrival", "makespan", "soc", "collisions"), mine, ref):
        assert np.array_equal(x, y), (name, [sample[i] for i in np.flatnonzero((x != y).reshape(len(sample), -1).any(1))]
                                      if name != "actions" else None)


def _sample(col, k, rng, per=1):
    """k random environments, and up to `per` each of: passed through (-2), no path (-1), repaired (0), unrepaired (> 0)."""
    B = len(col)
    out = set(rng.choice(B, size=min(k, B), replace=False).tolist())
    for sel in (col == -2, col == -1, col == 0, col > 0):
        out |= set(np.flatnonzero(sel)[:per].tolist())
    return sorted(out)


@pytest.mark.parametrize("B,N,L,H", [(512, 32, 40, 256), (64, 64, 80, 256), (512, 8, 20, 14)])
def test_parity_generated(B, N, L, H):
    rng = np.random.default_rng(B + N + L)
    env = _generated(B, N, L, seed=N + L)
    state = _state(env)
    seen = set()
    for source in ("plan", "plan_orders"):
        plan = env.plan(H) if source == "plan" else env.plan_orders(H, 8, seed=3)
        inp_np = tuple(x.cpu().numpy() for x in plan[:2])
        failed = (inp_np[1] == -1).all(1)
        for k in (1, 4, 8, N):
            I, seed = (3, 11) if N < 64 else (2, 12)
            got = _repair_np(env, plan, I, k, seed)
            col = got[4]
            assert ((col == -2) == ~failed).all()
            assert np.array_equal(got[0][:, ~failed], inp_np[0][:, ~failed]) and np.array_equal(got[1][~failed], inp_np[1][~failed])
            seen |= set(np.unique(np.clip(col, -2, 1)).tolist())
            _check_parity(got, state, inp_np, I, k, seed, _sample(col, 1, rng))
    # at H = 14 the failed environments are the ones some agent cannot reach in time
    assert -2 in seen and (0 in seen if H == 256 else -1 in seen)


def test_parity_sized_levels():
    from mapf_rl_b200 import BatchedEnvironment
    torch = _torch()
    rng = np.random.default_rng(45)
    B = 1024
    env = BatchedEnvironment(B, 6, 40, sized=True)
    env.reset(seed=12, env_offset=0, density=0.3, levels=LEVELS)
    n, l = (x.cpu().numpy().astype(np.int64) for x in env.sizes)
    state = _state(env)
    per_level = [int(np.flatnonzero((n == a) & (l == b))[0]) for a, b in LEVELS]
    for H in (256, 12):
        inp = env.plan(H)
        # absent rows hold values no plan writes: kept where the environment is passed through, written as plan() writes
        # them where it is repaired
        absent = np.arange(6)[None, :] >= n[:, None]
        mask = torch.as_tensor(absent, device="cuda")
        actions, arrival = inp[0].clone(), inp[1].clone()
        arrival[mask] = 99
        actions[:, mask] = 7
        inp_np = (actions.cpu().numpy(), arrival.cpu().numpy())
        for k in (1, 4):
            got = _repair_np(env, (actions, arrival), 6, k, seed=5)
            col = got[4]
            through = col == -2
            assert (got[1][absent & through[:, None]] == 99).all() and (got[0][:, absent & through[:, None]] == 7).all()
            assert (got[1][absent & (col == 0)[:, None]] == 0).all() and (got[0][:, absent & ~through[:, None]] == 0).all()
            assert (got[1][absent & ((col == -1) | (col > 0))[:, None]] == -1).all()
            _check_parity(got, state, inp_np, 6, k, 5, sorted(set(per_level) | set(_sample(col, 8, rng))), n=n, l=l)


def test_same_as_plan_where_plan_solves():
    torch = _torch()
    B, N, L, H = 8192, 32, 40, 256
    env = _generated(B, N, L, seed=77)
    base = _np(env.plan(H))
    solved = base[2] >= 0
    actions = torch.zeros((H, B, N), dtype=torch.uint8, device="cuda")
    arrival = torch.full((B, N), -1, dtype=torch.int32, device="cuda")
    got = _repair_np(env, (actions, arrival), 16, 8)
    assert (got[4][solved] == 0).all()
    assert np.array_equal(got[0][:, solved], base[0][:, solved]) and np.array_equal(got[1][solved], base[1][solved])
    assert (got[4] >= -1).all() and (got[4][~solved] != -2).all()


@pytest.mark.parametrize("B,N,L", [(512, 32, 40), (64, 24, 60)])
def test_composition_and_replay(B, N, L):
    rng = np.random.default_rng(B + N + 2)
    env = _generated(B, N, L, seed=5 * B + N + 2)
    state = _state(env)
    plan = env.plan(256)
    rep = env.plan_repair(plan[0], plan[1], 32, 8, seed=4)
    col = rep[4].cpu().numpy()
    fixed = np.flatnonzero(col == 0)
    assert (len(fixed) > 0 or B < 512) and (plan[2].cpu().numpy()[fixed] == -1).all()
    # repaired environments are valid plan_lns input (accepted 0, never -2); passed-through ones are plan()'s plans
    lns = _np(env.plan_lns(rep[0], rep[1], 0, 8))
    assert (lns[4][(col == 0) | (col == -2)] == 0).all() and (lns[4][(col == -1) | (col > 0)] == -1).all()
    better = _np(env.plan_lns(rep[0], rep[1], 16, 8, seed=2))
    rep_np = _np(rep)
    ok = rep_np[3] >= 0
    assert (better[3][ok] <= rep_np[3][ok]).all() and (better[4][col == 0] >= 0).all()
    _check_rollout(env, rep_np[:3], state, (fixed[:3].tolist() if len(fixed) else []) + rng.choice(B, size=1).tolist())


def test_determinism_sharding_and_isolation():
    from mapf_rl_b200 import BatchedEnvironment
    torch = _torch()
    B, N, L, H, I, k, seed = 512, 32, 40, 256, 8, 4, 31
    env = _generated(B, N, L, seed=17)
    maps, pos, goals = _state(env)
    plan = env.plan(H)
    before = (env.agents_pos.clone(), env.goals_pos.clone(), env.steps.clone(), env.navi_map.clone())
    caller = (plan[0].clone(), plan[1].clone())
    whole = _repair_np(env, plan, I, k, seed)
    again = _repair_np(env, plan, I, k, seed)
    for x, y in zip(whole, again):
        assert np.array_equal(x, y)
    assert torch.equal(plan[0], caller[0]) and torch.equal(plan[1], caller[1])
    for x, y in zip(before, (env.agents_pos, env.goals_pos, env.steps, env.navi_map)):
        assert torch.equal(x, y)
    env.check()
    half = B // 2
    parts = []
    for off in (0, half):
        h = BatchedEnvironment(half, N, L)
        h.load(maps[off:off + half], pos[off:off + half], goals[off:off + half])
        parts.append(_np(h.plan_repair(plan[0][:, off:off + half].contiguous(), plan[1][off:off + half], I, k, seed, env_offset=off)))
    for i, x in enumerate(whole):
        assert np.array_equal(x, np.concatenate([p[i] for p in parts], axis=1 if i == 0 else 0)), i
    # zero iterations: the initial soft plan, repaired only where it has no collision
    z = _repair_np(env, plan, 0, k, seed)
    _check_parity(z, (maps, pos, goals), _np(plan[:2]), 0, k, seed, _sample(z[4], 2, np.random.default_rng(1)))
    assert (z[4][whole[4] == -2] == -2).all() and ((z[4] == 0) <= (whole[4] == 0)).all()
    # another seed draws other neighbourhoods
    other = _repair_np(env, plan, I, k, seed + 1)
    assert not all(np.array_equal(x, y) for x, y in zip(other, whole))


def test_arguments_and_scratch():
    from mapf_rl_b200 import _native
    torch = _torch()
    B, N = 64, 8
    env = _generated(B, N, 12, seed=1)
    lib, h, st = env._lib, env._h, env._stream()
    act = torch.zeros((1025, B, N), dtype=torch.uint8, device="cuda")
    arr = torch.full((B, N), -1, dtype=torch.int32, device="cuda")
    col = torch.zeros(B, dtype=torch.int32, device="cuda")
    pa, pr, pc = (C.c_void_p(x.data_ptr()) for x in (act, arr, col))
    for H, I, k, a, r, c in ((0, 1, 1, pa, pr, pc), (1025, 1, 1, pa, pr, pc), (16, -1, 1, pa, pr, pc), (16, (1 << 24) + 1, 1, pa, pr, pc),
                             (16, 1, 0, pa, pr, pc), (16, 1, N + 1, pa, pr, pc), (16, 1, 1, None, pr, pc), (16, 1, 1, pa, None, pc),
                             (16, 1, 1, pa, pr, None)):
        assert lib.mapf_env_plan_repair(h, H, I, k, 0, 0, a, r, c, st) == _native.MAPF_EINVAL
        assert b"mapf_env_plan_repair" in lib.mapf_last_error()
    with pytest.raises(AssertionError):
        env.plan_repair(act.to(torch.int32), arr)
    with pytest.raises(AssertionError):
        env.plan_repair(act, arr[:, :4])
    env.check()
    # the scratch: 10 tables where plan() keeps 6, plus the current and candidate paths, 4 bytes per agent and step
    env2 = _generated(B, N, 12, seed=1)
    plan = env2.plan(256)
    torch.cuda.synchronize()
    bytes_plan = env2.arena_bytes
    env2.plan_repair(plan[0], plan[1], 4, 4)
    torch.cuda.synchronize()
    # L = 12: RW = 1, RPL = 1, 32 words per table slice; B / 4 blocks of 4 warps either way
    assert env2.arena_bytes - bytes_plan == (B // 4) * 4 * (4 * 257 * 32 * 4 + 4 * N * 257)


def test_golden_64():
    from mapf_rl_b200 import BatchedEnvironment
    maps, pos, goals = instances(64)
    env = BatchedEnvironment(len(maps), 64, 40)
    env.load(maps, pos, goals)
    plan = _np(env.plan(256))
    failed = plan[2] < 0
    got = _np(env.plan_repair(*(_torch().as_tensor(x).cuda() for x in plan[:2]), 64, 8))
    assert failed.sum() == 96 and (got[4][failed] == 0).sum() >= 85 and (got[4][~failed] == -2).all()


def _cbs_check(maps, pos, goals, N, L, node_limit):
    from mapf_rl_b200 import BatchedEnvironment, search
    env = BatchedEnvironment(len(maps), N, L)
    env.load(maps, pos, goals)
    dist = env.heuristic_distances().cpu().numpy()
    torch = _torch()
    B = len(maps)
    empty = (torch.zeros((256, B, N), dtype=torch.uint8, device="cuda"), torch.full((B, N), -1, dtype=torch.int32, device="cuda"))
    got = _repair_np(env, empty, 32, min(8, N), seed=1)
    _, T, cost, _ = search.solve_batch(maps, pos, goals, dist=dist, time_limit_s=0, node_limit=node_limit)
    both = (got[4] == 0) & (T >= 0)
    assert (got[3][both] >= cost[both]).all()
    return int(both.sum())


def test_against_cbs():
    both = 0
    for k, (L, N, density) in enumerate(CBS_CASES):
        m, s, g = cbs_instance(k, L, N, density)
        both += _cbs_check(m[None].astype(np.uint8), s[None].astype(np.uint8), g[None].astype(np.uint8), N, L, 1 << 16)
    maps, pos, goals = instances(16)
    both += _cbs_check(maps, pos, goals, 16, 40, 2000)
    assert both >= 20
