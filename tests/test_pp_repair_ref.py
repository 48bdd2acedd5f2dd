"""CPU self-checks of the restatement of plan repair (tests/pp_repair_ref.py): on an environment prioritized planning solves,
repairing its failed row gives pp_ref.plan's plan; the corridor instance index order cannot solve is repaired; the collision
identity and a never-increasing G on random instances (asserted inside the restatement); every repaired plan is a valid plan;
the collision cap and a short horizon give -1; a plan that is not failed is passed through with -2."""
import numpy as np

import pp_lns_ref
import pp_ref
import pp_repair_ref
from helpers import instances, random_instance


def _failed_row(N, H):
    return np.zeros((H, N), dtype=np.uint8), np.full(N, -1, dtype=np.int32)


def _valid(m, s, g, acts, arr, n=None):
    n = len(s) if n is None else n
    return pp_lns_ref.paths_of(m, np.asarray(s)[:n], np.asarray(g)[:n], acts[:, :n], arr[:n], n, m.shape[0]) is not None


def test_equals_plan_where_plan_solves():
    rng = np.random.default_rng(3)
    checked = 0
    while checked < 12:
        L, N = int(rng.integers(5, 10)), int(rng.integers(2, 8))
        m, s, g = random_instance(rng, L, N, 0.25)
        acts, arr = pp_ref.plan(m, s, g, 32)
        if (arr < 0).any():
            continue
        got = pp_repair_ref.plan_repair(m, s, g, *_failed_row(N, 32), 4, 2, 0, checked)
        assert got[2] == 0 and got[3] == 0 and np.array_equal(got[0], acts) and np.array_equal(got[1], arr)
        checked += 1
    maps, pos, goals = instances(16)
    golden = 0
    for e in range(len(maps)):
        acts, arr = pp_ref.plan(maps[e], pos[e], goals[e], 256)
        if (arr < 0).any():
            continue
        got = pp_repair_ref.plan_repair(maps[e], pos[e], goals[e], *_failed_row(16, 256), 8, 8, 0, e)
        assert got[2] == 0 and np.array_equal(got[0], acts) and np.array_equal(got[1], arr), e
        golden += 1
        if golden == 2:
            break


def test_corridor_repaired():
    m, s, g = pp_ref.corridor_instance()
    acts, arr = pp_ref.plan(m, s, g, 16)
    assert (arr == -1).all()
    history = []
    out_a, out_r, col, run = pp_repair_ref.plan_repair(m, s, g, acts, arr, 8, 2, 0, 0, history=history)
    assert col == 0 and 1 <= run <= 8 and history[0] > 0 and history[-1] == 0
    assert _valid(m, s, g, out_a, out_r)


def test_identity_monotone_and_validity():
    """Random crowded instances: the restatement asserts G(plan) = G(X) + f_new after every accepted iteration; G never
    increases, and every repaired plan is a valid plan."""
    rng = np.random.default_rng(11)
    repaired = started = 0
    for trial in range(40):
        L, N = int(rng.integers(5, 8)), int(rng.integers(4, 10))
        m, s, g = random_instance(rng, L, N, 0.3)
        if (pp_ref.plan(m, s, g, 24)[1] >= 0).all():
            continue
        history = []
        k = int(rng.integers(1, N + 1))
        out_a, out_r, col, run = pp_repair_ref.plan_repair(m, s, g, *_failed_row(N, 24), 12, k, trial, trial, history=history)
        if col == -1:
            continue
        started += 1
        assert all(b <= a for a, b in zip(history, history[1:])) and history[-1] == max(col, 0)
        assert len(history) == run + 1 and (run == 12 or history[-1] == 0)
        if col == 0:
            repaired += 1
            assert _valid(m, s, g, out_a, out_r)
            assert (out_a[np.arange(24)[:, None] >= out_r[None]] == 0).all()
        else:
            assert (out_r == -1).all() and not out_a.any()
    assert started >= 10 and repaired >= 5


def test_absent_agents_and_pass_through():
    rng = np.random.default_rng(5)
    m, s, g = random_instance(rng, 7, 6, 0.2)
    n = 4
    acts, arr = _failed_row(6, 32)
    arr[n:] = 77  # absent rows: only the present ones decide that the plan failed
    acts[:, n:] = 3
    out_a, out_r, col, _ = pp_repair_ref.plan_repair(m, s, g, acts, arr, 8, 2, 1, 0, n=n)
    assert col == 0 and (out_r[n:] == 0).all() and not out_a[:, n:].any() and _valid(m, s, g, out_a, out_r, n=n)
    # a plan that is not failed comes back as it went in, whether it is valid or not
    bad_a, bad_r = out_a.copy(), out_r.copy()
    bad_a[0, 0] = 5
    for a_in, r_in in ((out_a, out_r), (bad_a, bad_r)):
        got = pp_repair_ref.plan_repair(m, s, g, a_in, r_in, 8, 2, 1, 0, n=n)
        assert got[2] == -2 and np.array_equal(got[0], a_in) and np.array_equal(got[1], r_in)


def _parked_line(parked):
    """A one-row corridor: agents 0 .. parked-1 stand on their goals (0, 1 .. parked), the last agent crosses from (0, 0)
    to (0, parked + 1) through all of them."""
    L = parked + 2
    m = np.ones((L, L), dtype=np.uint8)
    m[0, :] = 0
    s = [[0, c] for c in range(1, parked + 1)] + [[0, 0]]
    g = [[0, c] for c in range(1, parked + 1)] + [[0, parked + 1]]
    return m, np.array(s, dtype=np.uint8), np.array(g, dtype=np.uint8)


def test_collision_cap():
    C = pp_repair_ref.MAX_COLLISIONS
    m, s, g = _parked_line(C + 1)  # C + 1 collisions at least
    assert pp_repair_ref.plan_repair(m, s, g, *_failed_row(len(s), 40), 4, 2, 0, 0)[2] == -1
    m, s, g = _parked_line(C)  # exactly C: a path, and collisions no group can remove in a corridor
    out = pp_repair_ref.plan_repair(m, s, g, *_failed_row(len(s), 40), 4, 2, 0, 0)
    assert out[2] > 0 and (out[1] == -1).all()


def test_short_horizon():
    m = np.zeros((5, 5), dtype=np.uint8)
    s, g = np.array([[0, 0], [4, 0]], dtype=np.uint8), np.array([[4, 4], [4, 1]], dtype=np.uint8)
    assert pp_repair_ref.plan_repair(m, s, g, *_failed_row(2, 7), 4, 2, 0, 0)[2] == -1  # agent 0 needs 8 steps
    assert pp_repair_ref.plan_repair(m, s, g, *_failed_row(2, 8), 4, 2, 0, 0)[2] == 0
