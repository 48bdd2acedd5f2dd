"""Plain numpy restatement of prioritized planning over several priority orders, `plan_orders_kernel`
(mapf_rl_b200/csrc/mapf_plan_kernels.cu, mapf_env_plan_prioritized_orders).  The rules (DESIGN.md §8 (f)5):

* Environment e of a handle has global index g = env_offset + e and n agents (N, or n_e on a sized handle).
* Order 0 is index order.  Order r >= 1 sorts the agents a < n by (k_a, a) ascending, k_a = word 0 of Philox4x32-10 with
  counter (g_lo, g_hi, PURPOSE_ORDER | r << 8, a) and key (seed_lo, seed_hi) -- the counter convention of the generator
  (tests/generator_ref.py), so the order depends on g and not on e.
* Planning in order pi is pp_ref.plan on the instance with its first n agents permuted by pi, the results un-permuted.
* The result is the solved order with the smallest sum of costs, ties to the smallest r: its actions and arrivals, order =
  r (-1 if every order fails) and rank[a] = agent a's position in it (255 for absent agents and failed environments).  A
  failed environment has arrival row -1 and all actions 0, as in pp_ref.plan.
"""
import numpy as np

import generator_ref
import pp_ref

PURPOSE_ORDER = 4
M32 = 0xFFFFFFFF


def priority_order(seed, g, r, n):
    """Order r of environment g: int64 [n], the agent at each position."""
    if r == 0:
        return np.arange(n, dtype=np.int64)
    idx = np.arange(n, dtype=np.uint64)
    key = generator_ref.philox4x32_10(g & M32, g >> 32, PURPOSE_ORDER | (r << 8), idx, seed & M32, seed >> 32)[0]
    return np.lexsort((idx, key)).astype(np.int64)


def plan_in_order(map_, starts, goals, horizon, perm, n=None, l=None):
    """pp_ref.plan with the first n agents taken in the order `perm`; results indexed by agent: (actions [H, N], arrival [N])."""
    starts, goals = np.asarray(starts), np.asarray(goals)
    N = starts.shape[0]
    n = N if n is None else int(n)
    s, g = starts.copy(), goals.copy()
    s[:n], g[:n] = starts[perm], goals[perm]
    acts, arr = pp_ref.plan(map_, s, g, horizon, n, l)
    actions, arrival = acts.copy(), arr.copy()
    actions[:, perm], arrival[perm] = acts[:, :n], arr[:n]
    return actions, arrival


def plan_orders(map_, starts, goals, horizon, orders, seed, g, n=None, l=None):
    """One environment of global index g: (actions uint8 [H, N], arrival int32 [N], order int, rank uint8 [N])."""
    N = np.asarray(starts).shape[0]
    n = N if n is None else int(n)
    best = None
    for r in range(orders):
        perm = priority_order(seed, g, r, n)
        actions, arrival = plan_in_order(map_, starts, goals, horizon, perm, n, l)
        if (arrival < 0).any():
            continue
        soc = int(arrival.sum())
        if best is None or soc < best[0]:
            best = (soc, r, perm, actions, arrival)
    rank = np.full(N, 255, dtype=np.uint8)
    if best is None:
        return np.zeros((int(horizon), N), dtype=np.uint8), np.full(N, -1, dtype=np.int32), -1, rank
    _, r, perm, actions, arrival = best
    rank[perm] = np.arange(n)
    return actions, arrival, r, rank


def plan_orders_batch(maps, starts, goals, horizon, orders, seed=0, env_offset=0, n=None, l=None, envs=None):
    """Environments `envs` (default all) of a batch: (actions uint8 [H, B', N], arrival int32 [B', N], makespan int32 [B'],
    soc int32 [B'], order int32 [B'], rank uint8 [B', N]); makespan and soc are -1 for a failed environment."""
    envs = range(len(maps)) if envs is None else envs
    res = [plan_orders(maps[e], starts[e], goals[e], horizon, orders, seed, env_offset + e, None if n is None else n[e],
                       None if l is None else l[e]) for e in envs]
    actions = np.stack([x[0] for x in res], axis=1)
    arrival = np.stack([x[1] for x in res])
    failed = (arrival < 0).any(1)
    makespan = np.where(failed, -1, arrival.max(1)).astype(np.int32)
    soc = np.where(failed, -1, arrival.sum(1)).astype(np.int32)
    return actions, arrival, makespan, soc, np.array([x[2] for x in res], dtype=np.int32), np.stack([x[3] for x in res])
