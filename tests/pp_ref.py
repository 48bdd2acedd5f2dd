"""Plain numpy restatement of the device prioritized planner, `plan_pp_kernel` (mapf_rl_b200/csrc/mapf_plan_kernels.cu).

The planner is deterministic, so every environment's plan can be compared with this one exactly.  The rules as the kernel
implements them (DESIGN.md §8 (f)5):

* Agents a = 0 .. n-1 are planned in index order over t = 0 .. H.  The committed paths of agents 0 .. a-1 define
  Occ(t) (cells they occupy at t; an agent parks on its goal from its arrival to H), SB_k(t) (cells v from which one of them
  moves to v - delta_k between t and t+1) and last_busy(c) (the largest t with c in Occ(t), or -1).
* F(0) = {start};  F(t+1) = (F(t) | OR_k (shift_k F(t) & ~SB_k(t))) & Free & ~Occ(t+1), where shift_k moves every cell by
  delta_k of action k (environment.py:12) and Free is the obstacle-free cells of the l x l map.
* arrival t* = min {t <= H : goal in F(t), t > last_busy(goal)}.  None (or an empty F) fails the environment: arrival row
  -1, every action 0, the remaining agents are not planned.
* back from (goal, t*) to t = 1: at (v, t) the first action k whose predecessor u = v - delta_k is in F(t-1) and, for a
  move, v is not in SB_k(t-1); actions[t-1, a] = k.  Actions from t* on are 0.
* commit: p_t into Occ(t) for t <= t*, the goal into Occ(t) for t* <= t <= H, and p_t into SB_opposite(k)(t) for every move
  p_t -> p_t+1 by action k.
* absent agents (a >= n) get arrival 0 and actions 0.
"""
import numpy as np

DELTA = ((0, 0), (-1, 0), (1, 0), (0, -1), (0, 1))
OPPOSITE = (0, 2, 1, 4, 3)


def shift(f, k):
    """out[v] = f[v - delta_k]: the cells reached from f by action k."""
    dx, dy = DELTA[k]
    out = np.zeros_like(f)
    L = f.shape[0]
    out[max(dx, 0):L + min(dx, 0), max(dy, 0):L + min(dy, 0)] = f[max(-dx, 0):L + min(-dx, 0), max(-dy, 0):L + min(-dy, 0)]
    return out


def plan(map_, starts, goals, horizon, n=None, l=None):
    """One environment: map_ [L, L] (non-zero = obstacle), starts / goals [N, 2]; n agents present (default N) on the
    l x l map (default L).  Returns (actions uint8 [H, N], arrival int32 [N])."""
    m = np.asarray(map_) != 0
    L = m.shape[0]
    starts, goals = np.asarray(starts, dtype=np.int64), np.asarray(goals, dtype=np.int64)
    N = starts.shape[0]
    n = N if n is None else int(n)
    l = L if l is None else int(l)
    H = int(horizon)
    free = ~m
    free[l:, :] = False
    free[:, l:] = False
    occ = np.zeros((H + 1, L, L), dtype=bool)
    sb = np.zeros((5, H + 1, L, L), dtype=bool)
    actions = np.zeros((H, N), dtype=np.uint8)
    arrival = np.zeros(N, dtype=np.int32)
    for a in range(n):
        (sx, sy), (gx, gy) = starts[a], goals[a]
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
            return np.zeros((H, N), dtype=np.uint8), np.full(N, -1, dtype=np.int32)
        path = [None] * (tstar + 1)
        vx, vy = int(gx), int(gy)
        path[tstar] = (vx, vy)
        for t in range(tstar, 0, -1):
            for k in range(5):
                ux, uy = vx - DELTA[k][0], vy - DELTA[k][1]
                if 0 <= ux < L and 0 <= uy < L and F[t - 1][ux, uy] and (k == 0 or not sb[k, t - 1, vx, vy]):
                    break
            else:
                raise AssertionError("no predecessor in the frontier history")
            actions[t - 1, a] = k
            vx, vy = ux, uy
            path[t - 1] = (vx, vy)
        for t, (x, y) in enumerate(path):
            occ[t, x, y] = True
            if t < tstar and actions[t, a]:
                sb[OPPOSITE[actions[t, a]], t, x, y] = True
        occ[tstar:, gx, gy] = True
        arrival[a] = tstar
    return actions, arrival


def corridor_instance():
    """5 x 5: a corridor along row 2 with a pocket at (1, 2).  Agent 0 steps from the pocket onto its goal (2, 2) in the
    corridor and parks there, on the only passage of agent 1 from (2, 0) to (2, 4): index order fails, though agent 1
    passing first and agent 0 stepping down after it solves the instance."""
    m = np.ones((5, 5), dtype=np.uint8)
    m[2, :] = 0
    m[1, 2] = 0
    return m, np.array([[1, 2], [2, 0]], dtype=np.uint8), np.array([[2, 2], [2, 4]], dtype=np.uint8)


def plan_batch(maps, starts, goals, horizon, n=None, l=None):
    """B environments: maps [B, L, L], starts / goals [B, N, 2], n / l optional [B].  Returns (actions uint8 [H, B, N],
    arrival int32 [B, N], makespan int32 [B], soc int32 [B]); makespan and soc are -1 for a failed environment."""
    B = len(maps)
    res = [plan(maps[i], starts[i], goals[i], horizon, None if n is None else n[i], None if l is None else l[i]) for i in range(B)]
    actions = np.stack([r[0] for r in res], axis=1)
    arrival = np.stack([r[1] for r in res])
    failed = (arrival < 0).any(1)
    makespan = np.where(failed, -1, arrival.max(1)).astype(np.int32)
    soc = np.where(failed, -1, arrival.sum(1)).astype(np.int32)
    return actions, arrival, makespan, soc
