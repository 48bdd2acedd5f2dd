"""Plain numpy restatement of plan improvement by large-neighbourhood search, `plan_lns_kernel`
(mapf_rl_b200/csrc/mapf_plan_kernels.cu, mapf_env_plan_lns).  The rules (DESIGN.md §8 (f)6):

* Input: a plan of the current state (map, positions as starts, goals) in `plan()`'s layout, actions [H, N] and arrival [N];
  H = actions.shape[0].  Environment e has global index g = env_offset + e, n agents and side l.
* Paths: agent a < n follows p_0 = start[a], p_t+1 = p_t + delta(actions[t, a]) for t < arrival[a], and p_t = goal[a] for
  arrival[a] <= t <= H.
* Input check, once: an arrival row of -1 (every present agent -1) is a failed plan, left unchanged with accepted -1.
  Otherwise the plan is left unchanged with accepted -2 if an action id is > 4, some p_t is outside the l x l map or on an
  obstacle, p_arrival[a] != goal[a], an action is non-zero at t >= arrival[a], arrival[a] is outside [0, H], two present
  agents share a cell at some t in [0, H], or two present agents swap cells between t and t + 1.  Rows of absent agents
  (a >= n) are neither read nor written.
* Iterations i = first_iteration .. first_iteration + I - 1: k_a = word 0 of Philox4x32-10 with counter
  (g_lo, g_hi, PURPOSE_LNS | i << 8, a) and key (seed_lo, seed_hi); the neighbourhood S is the m = min(k, n) agents of
  smallest (k_a, a), in that order.  The paths of the agents outside S are reserved in Occ / SB as pp_ref.plan commits a
  path, and the agents of S are planned in order by pp_ref.plan's rules (frontier, arrival after last_busy(goal), read-back
  to the lowest action id, commit) against them and against the agents of S planned before.  The iteration is accepted if
  every agent of S finds a path within H and the sum of their new arrivals is strictly less than the sum of their old ones:
  the new paths replace the old ones and accepted += 1.  Otherwise nothing changes.
* Output: the actions and arrivals of the final paths (actions 0 from an agent's arrival on) and accepted >= 0.  The result
  is valid input again, its sum of costs never exceeds the input's, and calls split by first_iteration give the result of
  one call over the same iterations.  With k >= n an iteration is plan_orders()'s planning in a fresh Philox order, kept
  only if strictly better.
"""
import numpy as np

import generator_ref
from pp_ref import DELTA, OPPOSITE, shift

PURPOSE_LNS = 5
M32 = 0xFFFFFFFF


def neighbourhood(seed, g, i, n, m):
    """S of iteration i in environment g: int64 [m], the m agents of smallest (k_a, a) in that order."""
    idx = np.arange(n, dtype=np.uint64)
    key = generator_ref.philox4x32_10(g & M32, g >> 32, PURPOSE_LNS | (i << 8), idx, seed & M32, seed >> 32)[0]
    return np.lexsort((idx, key))[:m].astype(np.int64)


def _move(u, v):
    """The action id of the move u -> v, 0 for a wait."""
    d = (v[0] - u[0], v[1] - u[1])
    return DELTA.index(d)


def paths_of(map_, starts, goals, actions, arrival, n, l):
    """The paths [n, H+1, 2] of a plan, or None if the plan is not valid (the input check's -2)."""
    m = np.asarray(map_) != 0
    H = actions.shape[0]
    paths = np.zeros((n, H + 1, 2), dtype=np.int64)
    for a in range(n):
        ar = int(arrival[a])
        if ar < 0 or ar > H:
            return None
        x, y = int(starts[a][0]), int(starts[a][1])
        for t in range(H + 1):
            if not (0 <= x < l and 0 <= y < l) or m[x, y]:
                return None
            if t == ar and (x, y) != (int(goals[a][0]), int(goals[a][1])):
                return None
            paths[a, t] = (x, y)
            if t == H:
                break
            k = int(actions[t, a])
            if k > 4 or (k and t >= ar):
                return None
            x, y = x + DELTA[k][0], y + DELTA[k][1]
    for t in range(H + 1):
        cells = {tuple(c) for c in paths[:, t]}
        if len(cells) < n:
            return None
        if t < H:
            moves = {(tuple(paths[a, t]), tuple(paths[a, t + 1])) for a in range(n) if (paths[a, t] != paths[a, t + 1]).any()}
            if any((v, u) in moves for u, v in moves):
                return None
    return paths


def _mark(occ, sb, path, value):
    """Path [H+1, 2] into (value True) or out of (False) the tables: p_t in Occ(t), p_t in SB_opposite(k)(t) for a move."""
    H = len(path) - 1
    for t in range(H + 1):
        x, y = path[t]
        occ[t, x, y] = value
        if t < H:
            k = _move(path[t], path[t + 1])
            if k:
                sb[OPPOSITE[k], t, x, y] = value


def plan_agent(free, occ, sb, start, goal, H):
    """pp_ref.plan's search and read-back for one agent against the reservations in occ / sb: (t*, path [H+1, 2] parked on
    the goal from t* on), or (-1, None)."""
    L = free.shape[0]
    (sx, sy), (gx, gy) = start, goal
    busy = np.flatnonzero(occ[:, gx, gy])
    lb = int(busy[-1]) if len(busy) else -1
    F = [np.zeros((L, L), dtype=bool)]
    F[0][sx, sy] = True
    tstar = -1
    if F[0][gx, gy] and 0 > lb:
        tstar = 0
    elif lb < H:
        for t in range(H):
            nf = F[t].copy()
            for k in range(1, 5):
                nf |= shift(F[t], k) & ~sb[k, t]
            nf &= free & ~occ[t + 1]
            F.append(nf)
            if not nf.any():
                break
            if nf[gx, gy] and t + 1 > lb:
                tstar = t + 1
                break
    if tstar < 0:
        return -1, None
    path = np.zeros((H + 1, 2), dtype=np.int64)
    path[tstar:] = (gx, gy)
    vx, vy = int(gx), int(gy)
    for t in range(tstar, 0, -1):
        for k in range(5):
            ux, uy = vx - DELTA[k][0], vy - DELTA[k][1]
            if 0 <= ux < L and 0 <= uy < L and F[t - 1][ux, uy] and (k == 0 or not sb[k, t - 1, vx, vy]):
                break
        else:
            raise AssertionError("no predecessor in the frontier history")
        vx, vy = ux, uy
        path[t - 1] = (vx, vy)
    return tstar, path


def plan_lns(map_, starts, goals, actions, arrival, iterations, neighborhood, seed, g, first_iteration=0, n=None, l=None):
    """One environment of global index g: (actions uint8 [H, N], arrival int32 [N], accepted int)."""
    m_ = np.asarray(map_) != 0
    L = m_.shape[0]
    starts, goals = np.asarray(starts, dtype=np.int64), np.asarray(goals, dtype=np.int64)
    actions, arrival = np.array(actions, dtype=np.uint8), np.array(arrival, dtype=np.int32)
    N = starts.shape[0]
    n = N if n is None else int(n)
    l = L if l is None else int(l)
    H = actions.shape[0]
    if (arrival[:n] == -1).all():
        return actions, arrival, -1
    paths = paths_of(m_, starts, goals, actions, arrival, n, l)
    if paths is None:
        return actions, arrival, -2
    free = ~m_
    free[l:, :] = False
    free[:, l:] = False
    occ = np.zeros((H + 1, L, L), dtype=bool)
    sb = np.zeros((5, H + 1, L, L), dtype=bool)
    for a in range(n):
        _mark(occ, sb, paths[a], True)
    arr = arrival[:n].astype(np.int64)
    m = min(int(neighborhood), n)
    accepted = 0
    for i in range(first_iteration, first_iteration + iterations):
        S = neighbourhood(seed, g, i, n, m)
        for a in S:
            _mark(occ, sb, paths[a], False)
        cand = []
        for a in S:
            tstar, path = plan_agent(free, occ, sb, starts[a], goals[a], H)
            if tstar < 0:
                break
            _mark(occ, sb, path, True)
            cand.append((tstar, path))
        if len(cand) == m and sum(c[0] for c in cand) < int(arr[S].sum()):
            for a, (tstar, path) in zip(S, cand):
                paths[a], arr[a] = path, tstar
            accepted += 1
        else:
            for _, path in cand:
                _mark(occ, sb, path, False)
            for a in S:
                _mark(occ, sb, paths[a], True)
    if accepted:
        for a in range(n):
            arrival[a] = arr[a]
            for t in range(H):
                actions[t, a] = _move(paths[a, t], paths[a, t + 1])
    return actions, arrival, accepted


def plan_lns_batch(maps, starts, goals, actions, arrival, iterations, neighborhood, seed=0, env_offset=0, first_iteration=0,
                   n=None, l=None, envs=None):
    """Environments `envs` (default all) of a batch, actions [H, B, N] and arrival [B, N] as plan() returns them:
    (actions uint8 [H, B', N], arrival int32 [B', N], makespan int32 [B'], soc int32 [B'], accepted int32 [B']); makespan
    and soc are -1 for a failed environment, derived as plan() derives them."""
    envs = range(len(maps)) if envs is None else envs
    res = [plan_lns(maps[e], starts[e], goals[e], actions[:, e], arrival[e], iterations, neighborhood, seed, env_offset + e,
                    first_iteration, None if n is None else n[e], None if l is None else l[e]) for e in envs]
    acts = np.stack([x[0] for x in res], axis=1)
    arr = np.stack([x[1] for x in res])
    failed = (arr < 0).any(1)
    makespan = np.where(failed, -1, arr.max(1)).astype(np.int32)
    soc = np.where(failed, -1, arr.sum(1)).astype(np.int32)
    return acts, arr, makespan, soc, np.array([x[2] for x in res], dtype=np.int32)
