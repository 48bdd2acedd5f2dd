"""CPU self-checks of the restatement of prioritized planning over several priority orders (tests/pp_orders_ref.py):
order 0 is pp_ref's index order, every order is a permutation whose plan replays collision-free through the oracle, the
best order never costs more than index order, and more orders solve instances index order cannot."""
import numpy as np

import pp_orders_ref
import pp_ref
from helpers import instances, random_instance
from oracle import oracle


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


def test_priority_order_is_a_permutation():
    for seed, g, r, n in [(0, 0, 1, 1), (0, 0, 0, 7), (5, 3, 1, 32), (7, 1 << 33, 255, 128), (2**64 - 1, 9, 17, 64)]:
        perm = pp_orders_ref.priority_order(seed, g, r, n)
        assert sorted(perm.tolist()) == list(range(n))
    assert pp_orders_ref.priority_order(1, 2, 0, 9).tolist() == list(range(9))
    # different orders, environments and seeds give different permutations
    base = pp_orders_ref.priority_order(1, 2, 3, 32).tolist()
    for args in [(1, 2, 4, 32), (1, 3, 3, 32), (2, 2, 3, 32)]:
        assert pp_orders_ref.priority_order(*args).tolist() != base


def test_one_order_is_index_order():
    rng = np.random.default_rng(11)
    for _ in range(20):
        L, N = int(rng.integers(4, 11)), int(rng.integers(1, 7))
        m, s, g = random_instance(rng, L, N, 0.2)
        n = int(rng.integers(1, N + 1))
        ra, rr = pp_ref.plan(m, s, g, 48, n=n)
        acts, arr, order, rank = pp_orders_ref.plan_orders(m, s, g, 48, 1, seed=3, g=int(rng.integers(0, 1000)), n=n)
        assert np.array_equal(acts, ra) and np.array_equal(arr, rr)
        if (rr >= 0).all():
            assert order == 0 and rank[:n].tolist() == list(range(n)) and (rank[n:] == 255).all()
        else:
            assert order == -1 and (rank == 255).all()


def test_every_order_replays_and_best_is_no_worse():
    rng = np.random.default_rng(12)
    R, H, better = 6, 64, 0
    for trial in range(30):
        L, N = int(rng.integers(4, 10)), int(rng.integers(2, 7))
        m, s, g = random_instance(rng, L, N, 0.2)
        socs = []
        for r in range(R):
            perm = pp_orders_ref.priority_order(trial, 5, r, N)
            acts, arr = pp_orders_ref.plan_in_order(m, s, g, H, perm)
            if (arr < 0).any():
                assert (arr == -1).all() and not acts.any()
                socs.append(None)
                continue
            _replay_ok(m, s, g, acts, int(arr.max()))
            for a in range(N):
                assert not acts[arr[a]:, a].any()
            socs.append(int(arr.sum()))
        acts, arr, order, rank = pp_orders_ref.plan_orders(m, s, g, H, R, trial, 5)
        solved = [x for x in socs if x is not None]
        if not solved:
            assert order == -1 and (arr == -1).all() and (rank == 255).all()
            continue
        assert order == socs.index(min(solved)) and int(arr.sum()) == min(solved)
        assert rank[pp_orders_ref.priority_order(trial, 5, order, N)].tolist() == list(range(N))
        if socs[0] is not None:
            assert min(solved) <= socs[0]
            better += min(solved) < socs[0]
        else:
            better += 1
    assert better >= 1


def _corridor_seed():
    """The first seed whose 8 orders solve the corridor instance that index order cannot."""
    m, s, g = pp_ref.corridor_instance()
    return next(seed for seed in range(32) if pp_orders_ref.plan_orders(m, s, g, 64, 8, seed, 0)[2] >= 0)


def test_corridor_solved_by_another_order():
    m, s, g = pp_ref.corridor_instance()
    assert pp_orders_ref.plan_orders(m, s, g, 64, 1, 0, 0)[2] == -1
    seed = _corridor_seed()
    acts, arr, order, rank = pp_orders_ref.plan_orders(m, s, g, 64, 8, seed, 0)
    assert order >= 1 and rank.tolist() == [1, 0] and arr.tolist() == [3, 4]
    _replay_ok(m, s, g, acts, 4)


def test_golden_64_more_orders_solve_more():
    maps, pos, goals = instances(64)
    k = 12
    one = pp_orders_ref.plan_orders_batch(maps[:k], pos[:k], goals[:k], 256, 1)
    eight = pp_orders_ref.plan_orders_batch(maps[:k], pos[:k], goals[:k], 256, 8)
    s1, s8 = one[2] >= 0, eight[2] >= 0
    assert (s8 >= s1).all() and s8.sum() > s1.sum()
    assert (eight[3][s1] <= one[3][s1]).all()
