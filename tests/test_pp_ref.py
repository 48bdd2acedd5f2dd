"""CPU self-checks of the prioritized-planning restatement (tests/pp_ref.py): hand-made cases with known answers, and plans
of random instances replayed through the oracle's Environment.step without a collision."""
import numpy as np

import pp_ref
from helpers import random_instance
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


def test_single_agent_is_shortest_path_and_horizon():
    m = np.zeros((6, 6), dtype=np.uint8)
    m[1:5, 2] = 1
    acts, arr = pp_ref.plan(m, [[2, 0]], [[2, 4]], 16)
    assert arr.tolist() == [8]          # around the wall: up 2 (or down 3), across 4, back 2
    moves = np.asarray(pp_ref.DELTA)[acts[:, 0]]
    assert (acts[:8, 0] != 0).all() and not acts[8:].any() and (moves.sum(0) == [0, 4]).all()
    acts, arr = pp_ref.plan(m, [[2, 0]], [[2, 4]], 7)
    assert arr.tolist() == [-1] and not acts.any()
    m[0, 2] = m[5, 2] = 1               # wall closed: unreachable
    assert pp_ref.plan(m, [[2, 0]], [[2, 4]], 64)[1].tolist() == [-1]
    assert pp_ref.plan(m, [[2, 0]], [[2, 0]], 4)[1].tolist() == [0]


def test_reservations_following_swap_and_parking():
    corridor = np.ones((5, 5), dtype=np.uint8)
    corridor[2, :] = 0
    # following a vacating agent is allowed: both move right in step 1
    acts, arr = pp_ref.plan(corridor, [[2, 1], [2, 0]], [[2, 2], [2, 1]], 8)
    assert arr.tolist() == [1, 1] and acts[0].tolist() == [4, 4]
    # head-on in a corridor: a swap is needed, so agent 1 fails
    acts, arr = pp_ref.plan(corridor, [[2, 0], [2, 4]], [[2, 4], [2, 0]], 32)
    assert arr.tolist() == [-1, -1] and not acts.any()
    # agent 0 parks on agent 1's only passage: index order fails, the other order solves it
    m, starts, goals = pp_ref.corridor_instance()
    acts, arr = pp_ref.plan(m, starts, goals, 32)
    assert arr.tolist() == [-1, -1] and not acts.any()
    acts, arr = pp_ref.plan(m, starts[::-1], goals[::-1], 32)
    assert arr.tolist() == [4, 3]
    # agent 0 crosses agent 1's goal at t = 2, so agent 1 arrives after that, at t = 3 and not 1
    acts, arr = pp_ref.plan(np.zeros((5, 5), dtype=np.uint8), [[1, 0], [0, 2]], [[1, 4], [1, 2]], 16)
    assert arr.tolist() == [4, 3] and acts[:4, 0].tolist() == [4, 4, 4, 4]
    # absent agents: arrival 0, no actions
    acts, arr = pp_ref.plan(corridor, [[2, 0], [2, 4]], [[2, 3], [2, 0]], 32, n=1)
    assert arr.tolist() == [3, 0] and not acts[:, 1].any()


def test_random_plans_replay_through_the_oracle():
    rng = np.random.default_rng(7)
    solved = 0
    for trial in range(40):
        L, N = int(rng.integers(4, 11)), int(rng.integers(1, 7))
        m, s, g = random_instance(rng, L, N, 0.2)
        acts, arr = pp_ref.plan(m, s, g, 64)
        if arr[0] < 0:
            assert (arr == -1).all() and not acts.any()
            continue
        solved += 1
        _replay_ok(m, s, g, acts, int(arr.max()))
        # an agent's actions stop at its arrival
        for a in range(N):
            assert not acts[arr[a]:, a].any()
    assert solved >= 15
