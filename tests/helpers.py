"""Shared test helpers: golden fixture access and action-stream generators."""
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def golden(name):
    return np.load(os.path.join(GOLDEN, name), allow_pickle=False)


_inst_cache = {}


def instances(num_agents):
    """-> maps uint8[200,40,40], agents uint8[200,N,2], goals uint8[200,N,2] (copy of test{N}_40_0.3.pkl)."""
    if "z" not in _inst_cache:
        z = golden("instances_40_0.3.npz")
        maps = np.unpackbits(z["maps_packed"], axis=1)[:, :1600].reshape(200, 40, 40).astype(np.uint8)
        _inst_cache["z"] = (z, maps)
    z, maps = _inst_cache["z"]
    return maps, z[f"agents{num_agents}"], z[f"goals{num_agents}"]


def greedy_actions(obs, rng, eps=0.1):
    """navi-greedy stream G for a batch: obs bool/uint8 [B,N,6,9,9] -> uint8 [B,N]."""
    B, N = obs.shape[:2]
    bits = obs[:, :, 2:6, 4, 4].astype(bool)                       # [B,N,4]
    score = rng.random((B, N, 4)) * bits                           # random tie-break among set bits
    act = np.where(bits.any(-1), 1 + score.argmax(-1), 0)
    explore = rng.random((B, N)) < eps
    act = np.where(explore, rng.integers(0, 5, size=(B, N)), act)
    return act.astype(np.uint8)


def random_instance(rng, L, N, density):
    """Unconstrained random instance (starts and goals distinct free cells, any component)."""
    while True:
        m = (rng.random((L, L)) < density).astype(np.uint8)
        free = np.argwhere(m == 0)
        if len(free) >= N:
            break
    a = free[rng.permutation(len(free))[:N]]
    g = free[rng.permutation(len(free))[:N]]
    return m, a.astype(np.uint8), g.astype(np.uint8)


# high-occupancy small boards (map_length, num_agents, density, seed): every conflict kind of environment.py:320-406 fires
RANDOM_GRID_CASES = [
    (3, 5, 0.0, 0), (3, 8, 0.0, 1), (4, 12, 0.0, 2), (4, 15, 0.0, 3), (5, 20, 0.0, 4), (6, 30, 0.0, 5),
    (6, 20, 0.15, 6), (8, 30, 0.2, 7), (10, 40, 0.3, 8), (12, 64, 0.1, 9), (2, 3, 0.0, 10), (2, 4, 0.0, 11),
]


def random_grid_trials(L, N, density, seed, trials=6, steps=40):
    """-> [(map, agents, goals, actions uint8[steps,N])] of one RANDOM_GRID_CASES entry: uniform actions, everybody
    moving, and moving with 20 % staying, in turn."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(trials):
        m, a, g = random_instance(rng, L, N, density)
        acts = np.empty((steps, N), dtype=np.uint8)
        for s in range(steps):
            mode = s % 3
            if mode == 0:
                acts[s] = rng.integers(0, 5, size=N)
            elif mode == 1:
                acts[s] = rng.integers(1, 5, size=N)          # everybody moves
            else:
                acts[s] = np.where(rng.random(N) < 0.2, 0, rng.integers(1, 5, size=N))
        out.append((m, a, g, acts))
    return out


# ---- instance-generator statistics (SURVEY 8f-3): the same numbers are computed for the live reference
# (tests/golden/make_golden.py -> generator_stats.npz), the host generator and the device generator ----
GEN_CONFIGS = [(20, 6), (12, 4)]  # (map_length, num_agents): the reference default (config.py) and a small, fragmented one


def _bfs_distance(free, s, g):
    """4-connected BFS distance between two free cells of the same component."""
    L = free.shape[0]
    dist = -np.ones((L, L), dtype=np.int32)
    dist[s[0], s[1]] = 0
    frontier = [(int(s[0]), int(s[1]))]
    while frontier:
        nxt = []
        for x, y in frontier:
            if x == g[0] and y == g[1]:
                return int(dist[x, y])
            for nx, ny in ((x - 1, y), (x + 1, y), (x, y - 1), (x, y + 1)):
                if 0 <= nx < L and 0 <= ny < L and free[nx, ny] and dist[nx, ny] < 0:
                    dist[nx, ny] = dist[x, y] + 1
                    nxt.append((nx, ny))
        frontier = nxt
    return -1


def generator_stats(maps, agents, goals):
    """Histograms (counts) of a batch of generated instances: realised obstacle density, start-goal BFS distance
    of every agent, size of agent 0's component relative to the free cells, number of distinct components the
    agents occupy.  Also checks the structural guarantees of environment.py:100-138 (distinct free cells,
    start and goal of an agent connected)."""
    from mapf_rl_b200.instances import map_partition
    maps, agents, goals = np.asarray(maps), np.asarray(agents).astype(np.int64), np.asarray(goals).astype(np.int64)
    B, L = maps.shape[0], maps.shape[1]
    N = agents.shape[1]
    dens = np.zeros(10, dtype=np.int64)            # density in [0, 0.5) by 0.05
    dist = np.zeros(2 * L, dtype=np.int64)          # BFS distance clipped to 2L-1
    comp = np.zeros(10, dtype=np.int64)            # |component of agent 0| / free cells, deciles
    ncomp = np.zeros(N + 1, dtype=np.int64)
    for k in range(B):
        m = maps[k] != 0
        free = ~m
        label, sizes = map_partition(m.astype(np.uint8))
        cells = np.concatenate([agents[k], goals[k]])
        assert free[cells[:, 0], cells[:, 1]].all(), "agent or goal on an obstacle"
        assert len({(int(x), int(y)) for x, y in cells}) == 2 * N, "starts and goals are not 2N distinct cells"
        la, lg = label[agents[k][:, 0], agents[k][:, 1]], label[goals[k][:, 0], goals[k][:, 1]]
        assert np.array_equal(la, lg), "start and goal in different components"
        dens[min(int(m.mean() / 0.05), 9)] += 1
        for i in range(N):
            d = _bfs_distance(free, agents[k][i], goals[k][i])
            assert d > 0
            dist[min(d, 2 * L - 1)] += 1
        comp[min(int(10 * sizes[la[0]] / max(int(free.sum()), 1)), 9)] += 1
        ncomp[len(set(la.tolist()))] += 1
    return {"density": dens, "distance": dist, "component": comp, "ncomponents": ncomp}


def histograms_agree(a, b, min_expected=8.0):
    """Two-sample chi-square on pooled bins (bins are merged left to right until both samples expect at least
    `min_expected`); returns the p-value."""
    from scipy.stats import chi2_contingency
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    ca, cb, acc_a, acc_b = [], [], 0.0, 0.0
    for x, y in zip(a, b):
        acc_a += x
        acc_b += y
        if min(acc_a, acc_b) >= min_expected:
            ca.append(acc_a), cb.append(acc_b)
            acc_a = acc_b = 0.0
    if ca:
        ca[-1] += acc_a
        cb[-1] += acc_b
    if len(ca) < 2:
        return 1.0
    return float(chi2_contingency(np.array([ca, cb]))[1])
