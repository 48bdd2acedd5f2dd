"""Plan improvement by large-neighbourhood search on the device (`BatchedEnvironment.plan_lns`, mapf_env_plan_lns): exact
parity with the numpy restatement (tests/pp_lns_ref.py) on generated batches, uniform and sized, from plan() and
plan_orders() output, with failed (-1), invalid (-2) and unimproved environments in every sample; replay through the rollout
kernel and the oracle; determinism, sharding by env_offset, calls split by first_iteration; the handle's state and the
caller's tensors unchanged; argument checks and the scratch in mapf_env_arena_bytes; and bounds against the project's CBS."""
import ctypes as C

import numpy as np
import pytest

import pp_lns_ref
from cbs_cases import CBS_CASES, cbs_instance
from helpers import instances
from test_gpu_plan_orders import LEVELS, _check_rollout
from test_pp_lns_ref import _invalid_cases

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


def _lns_np(env, plan, I, k, seed=0, env_offset=0, first=0):
    return _np(env.plan_lns(plan[0], plan[1], I, k, seed, env_offset, first))


def _corrupt(plan):
    """Makes the first two solved environments invalid input (an action id 5; an arrival past the horizon); returns the copy
    and the two environments."""
    envs = np.flatnonzero(plan[2].cpu().numpy() >= 0)[:2].tolist()
    actions, arrival = plan[0].clone(), plan[1].clone()
    actions[0, envs[0], 0] = 5
    arrival[envs[1], 0] = actions.shape[0] + 1
    return (actions, arrival), envs


def _check_parity(got, state, inp, I, k, seed, sample, n=None, l=None, env_offset=0, first=0):
    maps, pos, goals = state
    ref = pp_lns_ref.plan_lns_batch(maps, pos, goals, inp[0], inp[1], I, k, seed, env_offset, first, n, l, envs=sample)
    mine = [x[:, sample] if i == 0 else x[sample] for i, x in enumerate(got)]
    for name, x, y in zip(("actions", "arrival", "makespan", "soc", "accepted"), mine, ref):
        assert np.array_equal(x, y), (name, [sample[i] for i in np.flatnonzero((x != y).reshape(len(sample), -1).any(1))]
                                      if name != "actions" else None)


def _sample(acc, k, rng, per=2):
    """k random environments, and up to `per` each of: failed (-1), invalid (-2), unimproved (0), improved (> 0)."""
    B = len(acc)
    out = set(rng.choice(B, size=min(k, B), replace=False).tolist())
    for sel in (acc == -1, acc == -2, acc == 0, acc > 0):
        out |= set(np.flatnonzero(sel)[:per].tolist())
    return sorted(out)


# (N, L) = (32, 40), (64, 80), (8, 20); k in {1, 4, 8, N}; input from plan() and from plan_orders(); H = 256 with a few
# environments failed by a short horizon on the smallest maps
@pytest.mark.parametrize("B,N,L,H", [(512, 32, 40, 256), (64, 64, 80, 256), (512, 8, 20, 14)])
def test_parity_generated(B, N, L, H):
    torch = _torch()
    rng = np.random.default_rng(B + N + L)
    env = _generated(B, N, L, seed=N + L)
    state = _state(env)
    for source in ("plan", "plan_orders"):
        plan = env.plan(H) if source == "plan" else env.plan_orders(H, 8, seed=3)
        inp, bad = _corrupt(plan)
        inp_np = tuple(x.cpu().numpy() for x in inp)
        improved = 0
        for k in (1, 4, 8, N):
            I, seed = (8, 11) if N < 64 else (3, 12)
            got = _lns_np(env, inp, I, k, seed)
            acc = got[4]
            assert (acc[bad] == -2).all()
            assert (acc >= -2).all() and ((acc == -1) == (inp_np[1] == -1).all(1)).all()
            ok = acc >= 0
            assert (got[3][ok] <= inp_np[1][ok].sum(1)).all()
            improved += int((acc > 0).sum())
            _check_parity(got, state, inp_np, I, k, seed, _sample(acc, 3 if N < 64 else 1, rng, 2 if N < 64 else 1))
        # at H = 14 the solved environments are the easy ones: their plans are seldom improvable
        assert improved > 0 or H < 256
        torch.cuda.synchronize()


def test_parity_sized_levels():
    from mapf_rl_b200 import BatchedEnvironment
    rng = np.random.default_rng(44)
    B = 1024
    env = BatchedEnvironment(B, 6, 40, sized=True)
    env.reset(seed=12, env_offset=0, density=0.3, levels=LEVELS)
    n, l = (x.cpu().numpy().astype(np.int64) for x in env.sizes)
    state = _state(env)
    per_level = [int(np.flatnonzero((n == a) & (l == b))[0]) for a, b in LEVELS]
    for H in (256, 12):
        inp = env.plan_orders(H, 4, seed=2)
        # absent rows hold values no plan writes; they must come back as they went in
        absent = np.arange(6)[None, :] >= n[:, None]
        mask = _torch().as_tensor(absent, device="cuda")
        actions, arrival = inp[0].clone(), inp[1].clone()
        arrival[mask] = 99
        actions[:, mask] = 7
        inp_np = (actions.cpu().numpy(), arrival.cpu().numpy())
        for k in (1, 4):
            got = _lns_np(env, (actions, arrival), 6, k, seed=5)
            assert (got[1][absent] == 99).all() and (got[0][:, absent] == 7).all()
            _check_parity(got, state, inp_np, 6, k, 5, sorted(set(per_level) | set(_sample(got[4], 16, rng))), n=n, l=l)


@pytest.mark.parametrize("B,N,L", [(512, 32, 40), (64, 24, 60)])
def test_replay(B, N, L):
    rng = np.random.default_rng(B + N + 1)
    env = _generated(B, N, L, seed=5 * B + N + 1)
    state = _state(env)
    plan = env.plan(256)
    got = _lns_np(env, plan, 16, 8, seed=4)
    assert (got[4] > 0).any()
    _check_rollout(env, got[:3], state, rng.choice(B, size=3, replace=False).tolist())


def test_invalid_inputs_on_device():
    """The crafted invalid plans of the reference's tests (a vertex conflict, a swap, a wrong arrival, a move after arrival,
    into an obstacle, off the map, an action id of 5), one environment each, and the valid plan they come from."""
    from mapf_rl_b200 import BatchedEnvironment
    torch = _torch()
    cases = _invalid_cases()
    names = sorted(cases)
    base = cases["arrival_not_on_goal"][:4] + ([2, 2],)
    rows = [cases[x] for x in names] + [base]
    B = len(rows)
    maps = np.stack([r[0] for r in rows]).astype(np.uint8)
    pos, goals = (np.array([r[i] for r in rows], dtype=np.uint8) for i in (1, 2))
    actions = np.stack([r[3] for r in rows], axis=1)
    arrival = np.array([r[4] for r in rows], dtype=np.int32)
    env = BatchedEnvironment(B, 2, 5)
    env.load(maps, pos, goals)
    a_in, r_in = torch.as_tensor(actions).cuda(), torch.as_tensor(arrival).cuda()
    got = _lns_np(env, (a_in, r_in), 4, 2)
    assert got[4][:-1].tolist() == [-2] * (B - 1) and got[4][-1] >= 0, dict(zip(names, got[4].tolist()))
    assert np.array_equal(got[0][:, :-1], actions[:, :-1]) and np.array_equal(got[1][:-1], arrival[:-1])
    _check_parity(got, (maps, pos, goals), (actions, arrival), 4, 2, 0, list(range(B)))


def test_determinism_sharding_and_splits():
    from mapf_rl_b200 import BatchedEnvironment
    torch = _torch()
    B, N, L, H, I, k, seed = 512, 32, 40, 256, 12, 8, 31
    env = _generated(B, N, L, seed=17)
    maps, pos, goals = _state(env)
    plan = env.plan_orders(H, 4, seed=1)
    before = (env.agents_pos.clone(), env.goals_pos.clone(), env.steps.clone(), env.navi_map.clone())
    caller = (plan[0].clone(), plan[1].clone())
    whole = _lns_np(env, plan, I, k, seed)
    again = _lns_np(env, plan, I, k, seed)
    for x, y in zip(whole, again):
        assert np.array_equal(x, y)
    # the caller's tensors and the handle's state are untouched
    assert torch.equal(plan[0], caller[0]) and torch.equal(plan[1], caller[1])
    for x, y in zip(before, (env.agents_pos, env.goals_pos, env.steps, env.navi_map)):
        assert torch.equal(x, y)
    env.check()
    # two handles with env_offset give one handle's result
    half = B // 2
    parts = []
    for off in (0, half):
        h = BatchedEnvironment(half, N, L)
        h.load(maps[off:off + half], pos[off:off + half], goals[off:off + half])
        parts.append(_np(h.plan_lns(plan[0][:, off:off + half].contiguous(), plan[1][off:off + half], I, k, seed, env_offset=off)))
    for i, x in enumerate(whole):
        assert np.array_equal(x, np.concatenate([p[i] for p in parts], axis=1 if i == 0 else 0)), i
    # calls split by first_iteration give one call's result
    a = env.plan_lns(plan[0], plan[1], 5, k, seed)
    b = _np(env.plan_lns(a[0], a[1], I - 5, k, seed, first_iteration=5))
    for i in range(4):
        assert np.array_equal(b[i], whole[i]), i
    acc_a = a[4].cpu().numpy()
    ok = whole[4] >= 0
    assert np.array_equal(acc_a[ok] + b[4][ok], whole[4][ok]) and np.array_equal(b[4][~ok], whole[4][~ok])
    # zero iterations: the input, accepted 0 where it is a valid plan
    z = _lns_np(env, plan, 0, k, seed)
    assert np.array_equal(z[0], plan[0].cpu().numpy()) and np.array_equal(z[1], plan[1].cpu().numpy())
    assert ((z[4] == 0) | (z[4] == -1)).all()
    # another seed draws other neighbourhoods
    other = _lns_np(env, plan, I, k, seed + 1)
    assert not np.array_equal(other[1], whole[1])


def test_arguments_and_scratch():
    from mapf_rl_b200 import _native
    torch = _torch()
    B, N = 64, 8
    env = _generated(B, N, 12, seed=1)
    lib, h, st = env._lib, env._h, env._stream()
    act = torch.zeros((1025, B, N), dtype=torch.uint8, device="cuda")
    arr = torch.zeros((B, N), dtype=torch.int32, device="cuda")
    acc = torch.zeros(B, dtype=torch.int32, device="cuda")
    pa, pr, pc = (C.c_void_p(x.data_ptr()) for x in (act, arr, acc))
    for H, I, k, first, a, r, c in ((0, 1, 1, 0, pa, pr, pc), (1025, 1, 1, 0, pa, pr, pc), (16, -1, 1, 0, pa, pr, pc),
                                    (16, 1, 0, 0, pa, pr, pc), (16, 1, N + 1, 0, pa, pr, pc), (16, 2, 1, (1 << 24) - 1, pa, pr, pc),
                                    (16, 1, 1, 0, None, pr, pc), (16, 1, 1, 0, pa, None, pc), (16, 1, 1, 0, pa, pr, None)):
        assert lib.mapf_env_plan_lns(h, H, I, k, 0, 0, first, a, r, c, st) == _native.MAPF_EINVAL
        assert b"mapf_env_plan_lns" in lib.mapf_last_error()
    assert lib.mapf_env_plan_lns(h, 16, 1, N, 0, 0, (1 << 24) - 1, pa, pr, pc, st) == _native.MAPF_OK
    with pytest.raises(AssertionError):
        env.plan_lns(act.to(torch.int32), arr)
    with pytest.raises(AssertionError):
        env.plan_lns(act, arr[:, :4])
    with pytest.raises(AssertionError):
        env.plan_lns(act[:, :, :4], arr)
    env.check()
    # the scratch: plan()'s tables plus the current and candidate paths, 4 bytes per agent and step, per resident warp
    env2 = _generated(B, N, 12, seed=1)
    bytes0 = env2.arena_bytes
    plan = env2.plan(256)
    _torch().cuda.synchronize()
    bytes_plan = env2.arena_bytes
    env2.plan_lns(plan[0], plan[1], 4, 4)
    _torch().cuda.synchronize()
    bytes_lns = env2.arena_bytes
    # B / 4 blocks of 4 warps either way; each warp adds N x (H + 1) u16 twice
    assert bytes_plan > bytes0 and bytes_lns - bytes_plan == (B // 4) * 4 * 4 * N * 257


def _cbs_check(maps, pos, goals, N, L, node_limit):
    from mapf_rl_b200 import BatchedEnvironment, search
    env = BatchedEnvironment(len(maps), N, L)
    env.load(maps, pos, goals)
    dist = env.heuristic_distances().cpu().numpy()
    plan = env.plan(256)
    base_soc = plan[3].cpu().numpy()
    got = _lns_np(env, plan, 32, min(8, N), seed=1)
    soc = got[3]
    solved = base_soc >= 0
    assert np.array_equal(soc >= 0, solved) and (soc[solved] <= base_soc[solved]).all()
    _, T, cost, _ = search.solve_batch(maps, pos, goals, dist=dist, time_limit_s=0, node_limit=node_limit)
    both = solved & (T >= 0)
    assert (soc[both] >= cost[both]).all()
    return int(both.sum()), int((soc[solved] < base_soc[solved]).sum())


def test_against_cbs_cases():
    both = 0
    for k, (L, N, density) in enumerate(CBS_CASES):
        m, s, g = cbs_instance(k, L, N, density)
        b, _ = _cbs_check(m[None].astype(np.uint8), s[None].astype(np.uint8), g[None].astype(np.uint8), N, L, 1 << 16)
        both += b
    assert both >= 8


def test_against_cbs_golden_16():
    maps, pos, goals = instances(16)
    both, improved = _cbs_check(maps, pos, goals, 16, 40, 2000)
    assert both >= 20 and improved >= 1
