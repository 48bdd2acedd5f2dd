"""CPU self-checks of the restatement of plan improvement by large-neighbourhood search (tests/pp_lns_ref.py): with a
neighbourhood of every agent an iteration is prioritized planning in that iteration's Philox order, kept only if strictly
better; every output is a valid plan (an independent collision / goal check, and a replay through the oracle); the sum of
costs never increases; zero iterations change nothing; split calls give one call's result; invalid and failed input plans
are returned untouched with -2 and -1."""
import numpy as np
import pytest

import pp_lns_ref
import pp_orders_ref
import pp_ref
from helpers import random_instance
from oracle import oracle

DELTA = np.array(pp_ref.DELTA)


def _check_plan(m, starts, goals, actions, arrival, n=None):
    """Independent check of a plan: moves by ids 0 .. 4 on free cells, on the goal from the arrival on (no action after
    it), no shared cell and no swap at any step."""
    N = len(starts)
    n = N if n is None else n
    H = actions.shape[0]
    p = np.array(starts[:n], dtype=np.int64)
    seen = [p.copy()]
    for t in range(H):
        a = actions[t, :n].astype(np.int64)
        assert (a <= 4).all()
        assert not (a[t >= arrival[:n]]).any()
        p = p + DELTA[a]
        assert ((p >= 0) & (p < m.shape[0])).all() and not m[p[:, 0], p[:, 1]].any()
        seen.append(p.copy())
    P = np.stack(seen)  # [H+1, n, 2]
    for a in range(n):
        assert (P[arrival[a]:, a] == goals[a]).all()
    for t in range(H + 1):
        assert len({tuple(c) for c in P[t]}) == n, t
        if t < H:
            for a in range(n):
                for b in range(a + 1, n):
                    assert not ((P[t, a] == P[t + 1, b]).all() and (P[t, b] == P[t + 1, a]).all()), (t, a, b)


def _replay_ok(m, starts, goals, actions, makespan):
    env = oracle.OracleEnv()
    env.load(m, starts, goals)
    done = bool(np.array_equal(starts, goals))
    for t in range(makespan):
        assert not done
        (_, pos), rew, done, _ = env.step(np.asarray(actions[t], dtype=np.uint8))
        if t < makespan - 1:
            assert not done and min(rew) > -0.5 + 1e-6, (t, rew)
    assert done and np.array_equal(np.asarray(env.agents_pos), goals)


def _solved_instances(rng, count, H=48, density=0.2):
    out = []
    while len(out) < count:
        L, N = int(rng.integers(5, 10)), int(rng.integers(2, 7))
        m, s, g = random_instance(rng, L, N, density)
        acts, arr = pp_ref.plan(m, s, g, H)
        if (arr >= 0).all():
            out.append((m, s, g, acts, arr))
    return out


def test_whole_neighbourhood_is_a_chain_of_orders():
    rng = np.random.default_rng(21)
    improved = 0
    for trial, (m, s, g, acts, arr) in enumerate(_solved_instances(rng, 12)):
        N = len(s)
        I, seed, ge = 6, trial, 3 + trial
        out_a, out_r, acc = pp_lns_ref.plan_lns(m, s, g, acts, arr, I, N + 1, seed, ge)
        best_a, best_r, chain = acts, arr, 0
        for i in range(I):
            perm = pp_lns_ref.neighbourhood(seed, ge, i, N, N)
            assert sorted(perm.tolist()) == list(range(N))
            ca, cr = pp_orders_ref.plan_in_order(m, s, g, acts.shape[0], perm)
            if (cr >= 0).all() and cr.sum() < best_r.sum():
                best_a, best_r, chain = ca, cr, chain + 1
        assert acc == chain and np.array_equal(out_r, best_r) and np.array_equal(out_a, best_a)
        improved += acc > 0
    assert improved >= 1


@pytest.mark.parametrize("k", [1, 2, 3, 8])
def test_outputs_are_valid_plans_no_worse(k):
    rng = np.random.default_rng(100 + k)
    accepted = 0
    for trial, (m, s, g, acts, arr) in enumerate(_solved_instances(rng, 10, density=0.3)):
        out_a, out_r, acc = pp_lns_ref.plan_lns(m, s, g, acts, arr, 24, k, 7, trial)
        assert acc >= 0 and out_r.sum() <= arr.sum()
        assert (acc > 0) == (out_r.sum() < arr.sum())  # each accepted iteration lowers the sum of costs
        _check_plan(m, s, g, out_a, out_r)
        _replay_ok(m, s, g, out_a, int(out_r.max()))
        # the output is valid input again
        again = pp_lns_ref.plan_lns(m, s, g, out_a, out_r, 4, k, 8, trial)
        assert again[2] >= 0 and again[1].sum() <= out_r.sum()
        accepted += acc
    # one agent re-planned against all the others rarely finds better; larger groups do
    assert accepted >= 1 or k == 1


def test_absent_agents_untouched():
    rng = np.random.default_rng(5)
    m, s, g = random_instance(rng, 8, 6, 0.2)
    n = 4
    acts, arr = pp_ref.plan(m, s, g, 48, n=n)
    assert (arr[:n] >= 0).all()
    acts[:, n:] = 3  # absent rows are neither read nor written
    arr[n:] = 77
    out_a, out_r, acc = pp_lns_ref.plan_lns(m, s, g, acts, arr, 8, 2, 1, 0, n=n)
    assert acc >= 0 and (out_a[:, n:] == 3).all() and (out_r[n:] == 77).all()
    _check_plan(m, s, g, out_a, out_r, n=n)


def test_zero_iterations_is_identity_and_split_calls():
    rng = np.random.default_rng(9)
    for trial, (m, s, g, acts, arr) in enumerate(_solved_instances(rng, 8)):
        a0, r0, acc0 = pp_lns_ref.plan_lns(m, s, g, acts, arr, 0, 2, 3, trial)
        assert acc0 == 0 and np.array_equal(a0, acts) and np.array_equal(r0, arr)
        whole = pp_lns_ref.plan_lns(m, s, g, acts, arr, 9, 2, 3, trial)
        first = pp_lns_ref.plan_lns(m, s, g, acts, arr, 4, 2, 3, trial)
        second = pp_lns_ref.plan_lns(m, s, g, first[0], first[1], 5, 2, 3, trial, first_iteration=4)
        assert np.array_equal(whole[0], second[0]) and np.array_equal(whole[1], second[1])
        assert whole[2] == first[2] + second[2]


def _open(L=5):
    return np.zeros((L, L), dtype=np.uint8)


# (map, starts, goals, actions [H, N], arrival): each violates one rule of the input check
def _invalid_cases():
    H = 4
    cases = {}
    # agents 0 (0,1) -> (2,1) and 1 (1,0) -> (1,2) both stand on (1,1) at t = 1
    a = np.zeros((H, 2), dtype=np.uint8)
    a[:2, 0], a[:2, 1] = 2, 4
    cases["vertex"] = (_open(), [[0, 1], [1, 0]], [[2, 1], [1, 2]], a, [2, 2])
    # agents 0 (0,0) -> (0,1) and 1 (0,1) -> (0,0) swap between t = 0 and 1
    a = np.zeros((H, 2), dtype=np.uint8)
    a[0, 0], a[0, 1] = 4, 3
    cases["swap"] = (_open(), [[0, 0], [0, 1]], [[0, 1], [0, 0]], a, [1, 1])
    # a valid plan of two agents along rows 0 and 2, then one rule broken at a time
    a = np.zeros((H, 2), dtype=np.uint8)
    a[:2, :] = 4
    base = (_open(), [[0, 0], [2, 0]], [[0, 2], [2, 2]], a, [2, 2])
    cases["arrival_not_on_goal"] = base[:4] + ([1, 2],)
    cases["arrival_past_horizon"] = base[:4] + ([2, H + 1],)
    after = a.copy()
    after[3, 0] = 1
    cases["move_after_arrival"] = base[:3] + (after, [2, 2])
    blocked = _open()
    blocked[0, 1] = 1
    cases["obstacle"] = (blocked,) + base[1:]
    off = np.zeros((H, 2), dtype=np.uint8)
    off[0, 0], off[1, 0], off[:2, 1] = 1, 2, 4  # agent 0 steps to (-1, 0) and back
    cases["off_map"] = (_open(), [[0, 0], [2, 0]], [[0, 0], [2, 2]], off, [2, 2])
    bad = a.copy()
    bad[0, 1] = 5
    cases["action_5"] = base[:3] + (bad, [2, 2])
    return cases


def test_valid_base_case():
    m, s, g, a, r = _invalid_cases()["arrival_not_on_goal"][:4] + ([2, 2],)
    _check_plan(m, np.array(s), np.array(g), a, np.array(r))
    assert pp_lns_ref.plan_lns(m, s, g, a, r, 4, 1, 0, 0)[2] >= 0


@pytest.mark.parametrize("name", sorted(_invalid_cases()))
def test_invalid_inputs_untouched(name):
    m, s, g, a, r = _invalid_cases()[name]
    out_a, out_r, acc = pp_lns_ref.plan_lns(m, s, g, a, r, 8, 2, 0, 0)
    assert acc == -2 and np.array_equal(out_a, a) and np.array_equal(out_r, r)


def test_failed_row():
    m, s, g = pp_ref.corridor_instance()
    acts, arr = pp_ref.plan(m, s, g, 64)
    assert (arr == -1).all()
    out_a, out_r, acc = pp_lns_ref.plan_lns(m, s, g, acts, arr, 8, 2, 0, 0)
    assert acc == -1 and np.array_equal(out_a, acts) and np.array_equal(out_r, arr)


def test_batch_form():
    rng = np.random.default_rng(4)
    inst = _solved_instances(rng, 4, H=32)
    L = max(x[0].shape[0] for x in inst)
    N = max(len(x[1]) for x in inst)
    # pad every instance to L x L (obstacles) and N agents (absent), as a sized batch
    maps = np.ones((4, L, L), dtype=np.uint8)
    starts, goals = np.zeros((4, N, 2), dtype=np.uint8), np.zeros((4, N, 2), dtype=np.uint8)
    acts, arr = np.zeros((32, 4, N), dtype=np.uint8), np.zeros((4, N), dtype=np.int32)
    n, l = [], []
    for e, (m, s, g, a, r) in enumerate(inst):
        le, ne = m.shape[0], len(s)
        maps[e, :le, :le], starts[e, :ne], goals[e, :ne], acts[:, e, :ne], arr[e, :ne] = m, s, g, a, r
        n.append(ne), l.append(le)
    out = pp_lns_ref.plan_lns_batch(maps, starts, goals, acts, arr, 6, 2, 5, 10, n=n, l=l)
    for e, (m, s, g, a, r) in enumerate(inst):
        one = pp_lns_ref.plan_lns(m, s, g, a, r, 6, 2, 5, 10 + e)
        ne = len(s)
        assert np.array_equal(out[0][:, e, :ne], one[0]) and np.array_equal(out[1][e, :ne], one[1]) and out[4][e] == one[2]
        assert out[3][e] == one[1].sum() and out[2][e] == one[1].max()
