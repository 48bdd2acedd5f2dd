"""Plain numpy restatement of plan repair by collision-based large-neighbourhood search (MAPF-LNS2), `plan_repair_kernel`
(mapf_rl_b200/csrc/mapf_plan_kernels.cu, mapf_env_plan_repair).  The rules (DESIGN.md §8 (f)7):

* Input: a plan in `plan()`'s layout, actions [H, N] and arrival [N]; H = actions.shape[0].  Environment e has global index
  g = env_offset + e, n agents and side l.  Only a failed plan (arrival -1 for every present agent) is repaired; any other
  environment is passed through untouched with collisions -2.
* Conflicts: obstacles, the l x l bound and swaps (SB, as pp_ref.plan) are hard; vertex conflicts cost 1 each.
* Soft search of one agent against Occ / SB: layers c = 0 .. C (C = MAX_COLLISIONS); F_c(t) are the cells reached at t with
  exactly c vertex collisions and no fewer.  F_0(0) = {start};
  R_c(t) = (F_c(t) | OR_k (shift_k F_c(t) & ~SB_k(t))) & Free;
  F_c(t+1) = ((R_c(t) & ~Occ(t+1)) | (R_c-1(t) & Occ(t+1))) minus F_0(t+1) .. F_c-1(t+1).
  park(t) = #{t' in (t, H] : goal in Occ(t')}; the cost is min over t <= H of c(t) + park(t) with c(t) the layer holding
  the goal, t* the earliest t of that minimum; no layer holding the goal at any t means no path.  Read-back from
  (goal, t*, c(t*)): at (v, t, c), c' = c - [v in Occ(t)] and the first action id k whose predecessor v - delta_k is in
  F_c'(t-1) and, for a move, v is not in SB_k(t-1).
* Initial plan: every agent in index order by the soft search, each against the agents before it; an agent without a path
  gives collisions -1 and plan()'s failure form.  G is the vertex excess of the plan.
* Iterations i = 0 .. I-1 while G > 0: K = the agents with a vertex collision; k_a = word 0 of Philox4x32-10 with counter
  (g_lo, g_hi, PURPOSE_REPAIR | i << 8, a) and key (seed_lo, seed_hi); S = the first min(k, n) agents by ([a not in K], k_a, a).
  f_old = G - G(X) with X the agents outside S; S is re-planned in that order against X and the new paths of S before it,
  f_new = the sum of their costs.  Accepted if every agent of S finds a path and (f_new, sum of S's new arrivals) <
  (f_old, sum of the old ones): the paths are replaced and G = G - f_old + f_new.
* Output: G = 0 gives collisions 0 and the plan as plan() writes a solved environment; G > 0 gives collisions G and
  plan()'s failure form (arrival row -1, actions 0).
"""
import numpy as np

import generator_ref
from pp_ref import DELTA, OPPOSITE, shift

MAX_COLLISIONS = 15  # MAPF_PLAN_REPAIR_MAX_COLLISIONS
PURPOSE_REPAIR = 6
M32 = 0xFFFFFFFF


def _shift3(f, k):
    """shift_k of every layer of f [C, L, L]."""
    return shift(f.transpose(1, 2, 0), k).transpose(2, 0, 1)


def _moves(path):
    """The action ids of the moves path[t] -> path[t+1], int64 [H]."""
    d = path[1:] - path[:-1]
    return np.select([d[:, 0] == -1, d[:, 0] == 1, d[:, 1] == -1, d[:, 1] == 1], [1, 2, 3, 4], 0)


def commit(occ, sb, paths):
    """Paths [m, H+1, 2] into the tables as pp_ref.plan commits a path: p_t in Occ(t), p_t in SB_opposite(k)(t) for a move."""
    H = paths.shape[1] - 1
    t = np.arange(H + 1)
    opp = np.array(OPPOSITE)
    for p in paths:
        occ[t, p[:, 0], p[:, 1]] = True
        k = _moves(p)
        mv = k > 0
        sb[opp[k[mv]], t[:-1][mv], p[:-1, 0][mv], p[:-1, 1][mv]] = True


def excess(paths):
    """G: sum over t and cells of max(0, occupants - 1) for paths [m, H+1, 2]."""
    if len(paths) == 0:
        return 0
    key = paths[:, :, 0] * 256 + paths[:, :, 1] + 65536 * np.arange(paths.shape[1])[None]
    return int(key.size - len(np.unique(key)))


def colliding(paths):
    """K: bool [m], the agents that share a cell with another agent at some t."""
    key = paths[:, :, 0] * 256 + paths[:, :, 1] + 65536 * np.arange(paths.shape[1])[None]
    _, inv, cnt = np.unique(key.ravel(), return_inverse=True, return_counts=True)
    return (cnt[inv] > 1).reshape(key.shape).any(1)


def soft_search(free, occ, sb, start, goal, H):
    """(t*, path [H+1, 2] parked on the goal from t* on, cost) of one agent against occ / sb, or None."""
    C = MAX_COLLISIONS
    L = free.shape[0]
    (sx, sy), (gx, gy) = (int(start[0]), int(start[1])), (int(goal[0]), int(goal[1]))
    lay = np.full((H + 1, L, L), -1, dtype=np.int8)  # the layer of each cell at each t, -1 unreached
    lay[0, sx, sy] = 0
    busy = occ[:, gx, gy].astype(np.int64)
    park = np.cumsum(busy[::-1])[::-1] - busy  # park[t] = #{t' > t : goal in Occ(t')}
    best = None
    for t in range(H + 1):
        c = int(lay[t, gx, gy])
        if c >= 0 and (best is None or c + int(park[t]) < best[0]):
            best = (c + int(park[t]), t, c)
        top = int(lay[t].max())
        if t == H or top < 0:
            break
        cs = np.arange(min(top + 1, C) + 1)
        Fc = lay[t][None] == cs[:, None, None]  # F_c(t) for c = 0 .. min(top + 1, C)
        R = Fc.copy()
        for k in range(1, 5):
            R |= _shift3(Fc, k) & ~sb[k, t][None]
        R &= free[None]
        Rprev = np.concatenate([np.zeros((1, L, L), dtype=bool), R[:-1]])
        cand = (R & ~occ[t + 1][None]) | (Rprev & occ[t + 1][None])
        lay[t + 1] = np.where(cand.any(0), cand.argmax(0), -1)  # the lowest layer wins
    if best is None:
        return None
    cost, tstar, c = best
    path = np.zeros((H + 1, 2), dtype=np.int64)
    path[tstar:] = (gx, gy)
    vx, vy = gx, gy
    for t in range(tstar, 0, -1):
        cp = c - int(occ[t, vx, vy])
        for k in range(5):
            ux, uy = vx - DELTA[k][0], vy - DELTA[k][1]
            if 0 <= ux < L and 0 <= uy < L and lay[t - 1, ux, uy] == cp and (k == 0 or not sb[k, t - 1, vx, vy]):
                break
        else:
            raise AssertionError("no predecessor in the layer history")
        vx, vy, c = ux, uy, cp
        path[t - 1] = (vx, vy)
    assert c == 0 and (vx, vy) == (sx, sy)
    return tstar, path, cost


def neighbourhood(seed, g, i, in_k, m):
    """S of iteration i in environment g: int64 [m], the first m agents by ([a not in K], k_a, a)."""
    idx = np.arange(len(in_k), dtype=np.uint64)
    key = generator_ref.philox4x32_10(g & M32, g >> 32, PURPOSE_REPAIR | (i << 8), idx, seed & M32, seed >> 32)[0]
    return np.lexsort((idx, key, ~in_k))[:m].astype(np.int64)


def plan_repair(map_, starts, goals, actions, arrival, iterations, neighborhood, seed, g, n=None, l=None, history=None):
    """One environment of global index g: (actions uint8 [H, N], arrival int32 [N], collisions int, iterations run).
    Asserts the collision identity G(plan) = G(X) + f_new after every accepted iteration, and that G never increases;
    `history`, a list, receives G after the initial plan and after every iteration."""
    m_ = np.asarray(map_) != 0
    L = m_.shape[0]
    starts, goals = np.asarray(starts, dtype=np.int64), np.asarray(goals, dtype=np.int64)
    actions, arrival = np.array(actions, dtype=np.uint8), np.array(arrival, dtype=np.int32)
    N = starts.shape[0]
    n = N if n is None else int(n)
    l = L if l is None else int(l)
    H = actions.shape[0]
    if not (arrival[:n] == -1).all():
        return actions, arrival, -2, 0
    failed = (np.zeros((H, N), dtype=np.uint8), np.full(N, -1, dtype=np.int32))
    free = ~m_
    free[l:, :] = False
    free[:, l:] = False
    occ = np.zeros((H + 1, L, L), dtype=bool)
    sb = np.zeros((5, H + 1, L, L), dtype=bool)
    paths = np.zeros((n, H + 1, 2), dtype=np.int64)
    arr = np.zeros(n, dtype=np.int64)
    G = 0
    for a in range(n):
        r = soft_search(free, occ, sb, starts[a], goals[a], H)
        if r is None:
            return failed + (-1, 0)
        arr[a], paths[a], cost = r
        G += cost
        commit(occ, sb, paths[a:a + 1])
    assert G == excess(paths)
    if history is not None:
        history.append(G)
    m = min(int(neighborhood), n)
    run = 0
    for i in range(iterations):
        if G == 0:
            break
        run += 1
        S = neighbourhood(seed, g, i, colliding(paths), m)
        in_s = np.zeros(n, dtype=bool)
        in_s[S] = True
        occ[:] = False
        sb[:] = False
        commit(occ, sb, paths[~in_s])
        GX = excess(paths[~in_s])
        f_old = G - GX
        new = []
        for a in S:
            r = soft_search(free, occ, sb, starts[a], goals[a], H)
            if r is None:
                break
            new.append(r)
            commit(occ, sb, r[1][None])
        f_new = sum(r[2] for r in new)
        if len(new) == m and (f_new, sum(r[0] for r in new)) < (f_old, int(arr[S].sum())):
            for a, r in zip(S, new):
                arr[a], paths[a] = r[0], r[1]
            assert f_new <= f_old and excess(paths) == GX + f_new
            G = GX + f_new
        if history is not None:
            history.append(G)
    if G > 0:
        return failed + (G, run)
    actions[:] = 0
    arrival[:] = 0
    for a in range(n):
        arrival[a] = arr[a]
        actions[:, a] = _moves(paths[a])
    return actions, arrival, 0, run


def plan_repair_batch(maps, starts, goals, actions, arrival, iterations, neighborhood, seed=0, env_offset=0, n=None, l=None,
                      envs=None):
    """Environments `envs` (default all) of a batch, actions [H, B, N] and arrival [B, N] as plan() returns them:
    (actions uint8 [H, B', N], arrival int32 [B', N], makespan int32 [B'], soc int32 [B'], collisions int32 [B']); makespan
    and soc are -1 for a failed environment, derived as plan() derives them."""
    envs = range(len(maps)) if envs is None else envs
    res = [plan_repair(maps[e], starts[e], goals[e], actions[:, e], arrival[e], iterations, neighborhood, seed, env_offset + e,
                       None if n is None else n[e], None if l is None else l[e]) for e in envs]
    acts = np.stack([x[0] for x in res], axis=1)
    arr = np.stack([x[1] for x in res])
    failed = (arr < 0).any(1)
    makespan = np.where(failed, -1, arr.max(1)).astype(np.int32)
    soc = np.where(failed, -1, arr.sum(1)).astype(np.int32)
    return acts, arr, makespan, soc, np.array([x[2] for x in res], dtype=np.int32)
