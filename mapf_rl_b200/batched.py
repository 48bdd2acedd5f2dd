"""BatchedEnvironment — B lockstep MAPF environments resident on one B200.

The fast path of this package: torch CUDA tensors in, torch CUDA tensors out, every call one or two
launches of hand-written sm_100a kernels through the C ABI (include/mapf_b200.h).  Semantics per
environment are exactly the reference's `Environment` (environment.py:74-467); the drop-in single-env
class in `mapf_rl_b200.environment` is a B = 1 view of this one.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np

from . import _native, config


def _torch():
    import torch
    return torch


class BatchedEnvironment:
    OBS_SHAPE = config.obs_shape  # (6, 9, 9)

    def __init__(self, num_envs: int, num_agents: int = config.num_agents, map_length: int = config.map_length,
                 device=None, obs_radius: int = config.obs_radius, reward_fn: dict = config.reward_fn, sized: bool = False):
        """sized=True: every environment carries its own agent count n_e <= num_agents and map side l_e <= map_length
        (the reference's curriculum trains on a mix of settings, worker.py:424-425).  Agents a >= n_e are absent: their
        actions are ignored, their observation rows are zeros, their reward 0 (code 5), positions 255; cells outside l_e are
        off the map.  Agents a < n_e see exactly what a (n_e, l_e) handle gives.  `rollout`, `set_autoreset` and the
        host-buffer steps are not available on a sized handle."""
        torch = _torch()
        if not torch.cuda.is_available():
            raise RuntimeError("mapf_rl_b200 needs a CUDA device: the environment kernels have no CPU fallback")
        self._lib = _native.lib()
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.num_envs, self.num_agents, self.map_length = int(num_envs), int(num_agents), int(map_length)
        self.map_size = (self.map_length, self.map_length)
        self.obs_radius = int(obs_radius)
        self.reward_fn = dict(reward_fn)
        cfg = _native.EnvConfig(self.num_envs, self.num_agents, self.map_length, self.obs_radius, self.device.index,
                                (C.c_float * 5)(*[float(self.reward_fn[k]) for k in config.REWARD_ORDER]))
        h = C.c_void_p()
        _native.check(self._lib.mapf_env_create(C.byref(cfg), C.byref(h)))
        self._h = h
        self.sized = bool(sized)
        if self.sized:
            _native.check(self._lib.mapf_env_enable_sizes(h))
        B, N = self.num_envs, self.num_agents
        self._rewards = torch.empty((B, N), dtype=torch.float32, device=self.device)
        self._done = torch.empty((B,), dtype=torch.uint8, device=self.device)
        self._steps = torch.empty((B,), dtype=torch.int32, device=self.device)
        self._resets = 0

    # -- plumbing ------------------------------------------------------------------------------
    def close(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            self._lib.mapf_env_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return C.c_void_p(_torch().cuda.current_stream(self.device).cuda_stream)

    def _dev_u8(self, x, shape, as_mask=False):
        """Bring an array-like to a contiguous uint8 tensor on this device (as_mask: non-zero -> 1)."""
        torch = _torch()
        t = x if isinstance(x, torch.Tensor) else torch.as_tensor(np.ascontiguousarray(x))
        if as_mask:
            t = (t != 0)
        t = t.to(device=self.device, dtype=torch.uint8).contiguous()
        assert tuple(t.shape) == tuple(shape), f"expected shape {shape}, got {tuple(t.shape)}"
        return t

    def _coords_u8(self, x, shape):
        """Coordinates -> uint8 tensor on this device; anything outside [0, L) raises here instead of wrapping in the
        uint8 cast (the reference raises IndexError when it indexes the map with such a coordinate)."""
        torch = _torch()
        t = x if isinstance(x, torch.Tensor) else torch.as_tensor(np.ascontiguousarray(x))
        assert tuple(t.shape) == tuple(shape), f"expected shape {shape}, got {tuple(t.shape)}"
        if t.dtype != torch.uint8 or self.map_length < 256:
            lo, hi = (int(t.min()), int(t.max())) if t.numel() else (0, 0)
            if lo < 0 or hi >= self.map_length:
                raise IndexError(f"coordinate outside the {self.map_length}x{self.map_length} map: min {lo}, max {hi}")
        return t.to(device=self.device, dtype=torch.uint8).contiguous()

    @property
    def arena_bytes(self) -> int:
        return int(self._lib.mapf_env_arena_bytes(self._h))

    # -- Environment.load (environment.py:198-215) ----------------------------------------------
    def load(self, maps, agents_pos, goals_pos, env_ids=None, num_agents=None, map_length=None):
        """maps [n,L,L] (0 free / non-zero obstacle, any dtype), agents_pos / goals_pos [n,N,2].
        env_ids: which slots to load (default 0..n-1).  Recomputes the heuristic maps of those slots.
        Sized handle: num_agents / map_length [n] give each instance's setting (default N / L); map cells outside
        l_e x l_e and agent rows >= n_e are ignored, and a coordinate of a present agent >= l_e raises IndexError."""
        torch = _torch()
        L, N = self.map_length, self.num_agents
        n = int(maps.shape[0])
        m = self._dev_u8(maps, (n, L, L), as_mask=True)
        if num_agents is not None or map_length is not None:
            assert self.sized, "per-environment sizes need a sized handle (BatchedEnvironment(..., sized=True))"
            ns = np.broadcast_to(np.asarray(N if num_agents is None else num_agents, dtype=np.int64), (n,))
            ls = np.broadcast_to(np.asarray(L if map_length is None else map_length, dtype=np.int64), (n,))
            if n and (ns.min() < 1 or ns.max() > N or ls.min() < 2 or ls.max() > L):
                raise ValueError(f"sizes outside 1 <= num_agents <= {N}, 2 <= map_length <= {L}")
            a = self._coords_sized(agents_pos, ns, ls)
            g = self._coords_sized(goals_pos, ns, ls)
        else:
            a = self._coords_u8(agents_pos, (n, N, 2))
            g = self._coords_u8(goals_pos, (n, N, 2))
        ids_ptr = None
        if env_ids is not None:
            ids = torch.as_tensor(env_ids, dtype=torch.int32).to(self.device).contiguous()
            assert ids.numel() == n
            ids_ptr = C.c_void_p(ids.data_ptr())
        if num_agents is not None or map_length is not None:
            nd = torch.as_tensor(np.ascontiguousarray(ns, dtype=np.uint8)).to(self.device)
            ld = torch.as_tensor(np.ascontiguousarray(ls, dtype=np.uint8)).to(self.device)
            _native.check(self._lib.mapf_env_load_sized(self._h, ids_ptr, n, C.c_void_p(m.data_ptr()), C.c_void_p(a.data_ptr()),
                                                        C.c_void_p(g.data_ptr()), C.c_void_p(nd.data_ptr()),
                                                        C.c_void_p(ld.data_ptr()), self._stream()))
        else:
            _native.check(self._lib.mapf_env_load(self._h, ids_ptr, n, C.c_void_p(m.data_ptr()), C.c_void_p(a.data_ptr()),
                                                  C.c_void_p(g.data_ptr()), self._stream()))
        # synchronous (keeps the inputs alive until the stream has consumed them); raises IndexError if the device-side
        # validation found a coordinate outside the map / a slot id outside the batch, RuntimeError('unique') for two
        # agents on one cell (environment.py:424-428 raises that at the next step)
        self.check()

    def _coords_sized(self, x, ns, ls):
        """[n,N,2] coordinates of a sized load -> uint8 tensor on this device; rows a >= n_e are ignored (sent as 0), a
        present agent's coordinate outside [0, l_e) raises IndexError."""
        torch = _torch()
        n, N = len(ns), self.num_agents
        t = np.asarray(x.cpu() if isinstance(x, torch.Tensor) else x)
        assert t.shape == (n, N, 2), f"expected shape {(n, N, 2)}, got {t.shape}"
        present = np.arange(N)[None, :] < ns[:, None]
        t = np.where(present[..., None], t.astype(np.int64), 0)
        bad = present & ((t < 0) | (t >= ls[:, None, None])).any(-1)
        if bad.any():
            i, a = np.argwhere(bad)[0]
            raise IndexError(f"coordinate {tuple(t[i, a])} of agent {a} outside the {ls[i]}x{ls[i]} map of instance {i}")
        return torch.as_tensor(t.astype(np.uint8)).to(self.device).contiguous()

    @property
    def sizes(self):
        """(num_agents uint8[B], map_length uint8[B]) CUDA tensors: each environment's setting (sized handle)."""
        torch = _torch()
        assert self.sized, "sizes of a handle created without sized=True"
        n = torch.empty((self.num_envs,), dtype=torch.uint8, device=self.device)
        l = torch.empty((self.num_envs,), dtype=torch.uint8, device=self.device)
        _native.check(self._lib.mapf_env_get_sizes(self._h, C.c_void_p(n.data_ptr()), C.c_void_p(l.data_ptr()), self._stream()))
        return n, l

    # -- Environment.reset generator, device side (environment.py:146-196) ----------------------
    def reset(self, mask=None, seed: int = 0, env_offset: Optional[int] = None, density: Optional[float] = None, levels=None):
        """Draw new random instances on the device for slots with mask != 0 (default: all).  Slot e draws Philox stream
        (seed, env_offset + e).  Without an explicit `env_offset` the handle counts its resets and uses
        resets * num_envs, so repeated `reset(mask)` calls at episode ends never hand a slot the instance it (or another
        slot) had before; pass `env_offset` to pin the instances (sharding, reproducing a run).
        levels (sized handle): a sequence of (num_agents, map_length) settings; each reset slot draws one uniformly from its
        own stream and generates the instance a uniform handle of that setting draws for the stream.  Without `levels`
        a sized handle resets its slots to (N, L)."""
        if env_offset is None:
            env_offset = self._resets * self.num_envs
        self._resets += 1
        mptr = None
        if mask is not None:
            mk = self._dev_u8(mask, (self.num_envs,))
            mptr = C.c_void_p(mk.data_ptr())
        dens = -1.0 if density is None else float(density)
        if levels is not None:
            assert self.sized, "levels need a sized handle (BatchedEnvironment(..., sized=True))"
            lv = np.asarray(levels, dtype=np.int64).reshape(-1, 2)
            if lv.size == 0 or lv.min() < 0 or lv.max() > 255:
                raise ValueError(f"levels must be a non-empty list of (num_agents, map_length) pairs, got {levels!r}")
            ld = _torch().as_tensor(np.ascontiguousarray(lv, dtype=np.uint8)).to(self.device)
            _native.check(self._lib.mapf_env_reset_levels(self._h, mptr, C.c_uint64(seed), C.c_uint64(env_offset),
                                                          C.c_float(dens), C.c_void_p(ld.data_ptr()), int(lv.shape[0]),
                                                          self._stream()))
            return
        _native.check(self._lib.mapf_env_reset(self._h, mptr, C.c_uint64(seed), C.c_uint64(env_offset),
                                               C.c_float(dens), self._stream()))

    # -- Environment.step + observe (environment.py:278-467) -------------------------------------
    def step(self, actions, out_obs=None, out_rewards=None, out_done=None, obs_rows=None, out_codes=None, out_bits=None):
        """actions: uint8 CUDA tensor [B,N] (anything else is converted).
        Returns (obs uint8[B,N,6,9,9], rewards float32[B,N], done uint8[B]); obs is written into
        `out_obs` when given (e.g. a slot of a device replay tensor).  With `obs_rows` (int64 CUDA tensor [B]),
        `out_obs` is the whole observation buffer of a replay store ([rows,N,6,9,9]) and environment e writes
        its block at row obs_rows[e] (returned obs is then `out_obs` itself).  `out_codes` (uint8 CUDA tensor [B,N])
        additionally receives the reward codes (index into config.REWARD_ORDER).
        `out_bits` (uint8 CUDA tensor [rows,N,64], instead of `out_obs`): the observation is written PACKED
        (`mapf_rl_b200.packed`), at row obs_rows[e] or row e, and `out_bits` is returned in its place."""
        torch = _torch()
        B, N = self.num_envs, self.num_agents
        if not (isinstance(actions, torch.Tensor) and actions.dtype == torch.uint8 and actions.is_cuda
                and actions.is_contiguous()):
            actions = torch.as_tensor(np.asarray(actions) if not isinstance(actions, torch.Tensor) else actions)
            actions = actions.to(device=self.device, dtype=torch.uint8).contiguous()
        assert actions.shape == (B, N), "actions number"
        if out_bits is not None:
            assert out_obs is None, "out_bits replaces out_obs"
            rewards = out_rewards if out_rewards is not None else self._rewards
            done = out_done if out_done is not None else self._done
            _native.check(self._lib.mapf_env_step_observe_packed(
                self._h, C.c_void_p(actions.data_ptr()), C.c_void_p(out_bits.data_ptr()), self._bits_rows(out_bits, obs_rows),
                C.c_void_p(rewards.data_ptr()), self._codes_ptr(out_codes), C.c_void_p(done.data_ptr()),
                C.c_void_p(self._steps.data_ptr()), self._stream()))
            return out_bits, rewards, done
        obs = out_obs if out_obs is not None else torch.empty((B, N, *self.OBS_SHAPE), dtype=torch.uint8, device=self.device)
        rewards = out_rewards if out_rewards is not None else self._rewards
        done = out_done if out_done is not None else self._done
        rows_ptr = None
        if obs_rows is not None:
            assert out_obs is not None and obs.is_contiguous() and obs.dtype == torch.uint8 and obs.shape[1] == N
            assert obs_rows.dtype == torch.int64 and obs_rows.is_cuda and obs_rows.numel() == B
            rows_ptr = C.c_void_p(obs_rows.data_ptr())
        else:
            assert obs.is_contiguous() and obs.dtype == torch.uint8 and obs.numel() == B * N * 486
        codes_ptr = self._codes_ptr(out_codes)
        _native.check(self._lib.mapf_env_step_observe_ex(
            self._h, C.c_void_p(actions.data_ptr()), C.c_void_p(obs.data_ptr()), rows_ptr, C.c_void_p(rewards.data_ptr()),
            codes_ptr, C.c_void_p(done.data_ptr()), C.c_void_p(self._steps.data_ptr()), self._stream()))
        return obs, rewards, done

    def _codes_ptr(self, out_codes):
        if out_codes is None:
            return None
        torch = _torch()
        assert (out_codes.is_cuda and out_codes.dtype == torch.uint8 and out_codes.is_contiguous()
                and out_codes.numel() == self.num_envs * self.num_agents)
        return C.c_void_p(out_codes.data_ptr())

    def _bits_rows(self, bits, rows, row_bytes=64):
        """Checks a packed output buffer [rows, N, row_bytes] and its optional int64 row tensor [B]; -> row pointer."""
        torch = _torch()
        B, N = self.num_envs, self.num_agents
        assert (bits.is_cuda and bits.dtype == torch.uint8 and bits.is_contiguous() and bits.dim() == 3
                and tuple(bits.shape[1:]) == (N, row_bytes)), f"packed buffer must be uint8 [rows, {N}, {row_bytes}]"
        if rows is None:
            assert bits.shape[0] >= B
            return None
        assert rows.dtype == torch.int64 and rows.is_cuda and rows.is_contiguous() and rows.numel() == B
        return C.c_void_p(rows.data_ptr())

    def rollout(self, actions, num_steps: Optional[int] = None, out_obs=None, out_rewards=None, out_done=None,
                out_steps=None, chains: int = 0, out_codes=None):
        """`num_steps` lockstep steps with the actions already on the device (mapf_env_rollout): the loop
        `for t: env.step(actions[t])` of test.py:120-130 when the actions do not depend on the observations.
        actions uint8[A,B,N] (step t uses slot t % A; num_steps defaults to A); out_obs uint8[R,B,N,6,9,9],
        out_rewards float32[S,B,N], out_done uint8[S,B], out_steps int32[S,B] are rings indexed t % R / t % S
        (allocated with one slot per step when not given).  The batch runs as `chains` independent sub-batch chains
        on internal streams (0 = default: one launch of the persistent rollout kernel).  `out_codes` uint8[S,B,N]
        additionally receives reward codes; `out_rewards=False` skips the fp32 rewards (codes only).  Asynchronous on
        the current stream.  Returns (obs, rewards, done, steps) rings."""
        torch = _torch()
        B, N = self.num_envs, self.num_agents
        assert isinstance(actions, torch.Tensor) and actions.is_cuda and actions.dtype == torch.uint8 and actions.is_contiguous()
        assert actions.dim() == 3 and tuple(actions.shape[1:]) == (B, N), "actions number"
        A = int(actions.shape[0])
        T = A if num_steps is None else int(num_steps)
        obs = out_obs if out_obs is not None else torch.empty((T, B, N, *self.OBS_SHAPE), dtype=torch.uint8, device=self.device)
        if out_rewards is False:
            assert out_codes is not None, "out_rewards=False needs out_codes"
            rewards = None
            S = int(out_codes.shape[0])
        else:
            rewards = out_rewards if out_rewards is not None else torch.empty((T, B, N), dtype=torch.float32, device=self.device)
            S = int(rewards.shape[0])
        done = out_done if out_done is not None else torch.empty((S, B), dtype=torch.uint8, device=self.device)
        steps = out_steps if out_steps is not None else torch.empty((S, B), dtype=torch.int32, device=self.device)
        assert obs.is_contiguous() and obs.dtype == torch.uint8 and tuple(obs.shape[1:]) == (B, N, *self.OBS_SHAPE)
        assert rewards is None or (rewards.is_contiguous() and rewards.dtype == torch.float32 and tuple(rewards.shape) == (S, B, N))
        assert done.is_contiguous() and done.dtype == torch.uint8 and tuple(done.shape) == (S, B)
        assert steps.is_contiguous() and steps.dtype == torch.int32 and tuple(steps.shape) == (S, B)
        if out_codes is not None:
            assert out_codes.is_cuda and out_codes.is_contiguous() and out_codes.dtype == torch.uint8 and tuple(out_codes.shape) == (S, B, N)
        io = _native.RolloutIO(T, actions.data_ptr(), A, obs.data_ptr(), int(obs.shape[0]),
                               rewards.data_ptr() if rewards is not None else None,
                               out_codes.data_ptr() if out_codes is not None else None, done.data_ptr(), steps.data_ptr(), S,
                               int(chains))
        _native.check(self._lib.mapf_env_rollout_ex(self._h, C.byref(io), self._stream()))
        return obs, rewards, done, steps

    def plan(self, horizon: int = config.max_steps):
        """Prioritized planning on the device (mapf_env_plan_prioritized) from the current state: agents in index order,
        each on its earliest-arrival path that avoids the paths of the agents before it (no shared cell, no swap), parked
        on its goal afterwards.  Returns (actions uint8[H,B,N], arrival int32[B,N], makespan int32[B], soc int32[B]) CUDA
        tensors on the current stream.  `actions` is the [T, B, N] script `rollout` replays as it is.  arrival: each
        agent's arrival step, 0 for absent agents; makespan / soc are the maximum / sum of an environment's arrivals.  An
        environment where some agent finds no path within `horizon` steps has arrival row, makespan and soc -1 and all
        actions 0.  The handle's state is not changed."""
        torch = _torch()
        B, N, H = self.num_envs, self.num_agents, int(horizon)
        actions = torch.empty((max(H, 1), B, N), dtype=torch.uint8, device=self.device)
        arrival = torch.empty((B, N), dtype=torch.int32, device=self.device)
        _native.check(self._lib.mapf_env_plan_prioritized(self._h, H, C.c_void_p(actions.data_ptr()),
                                                          C.c_void_p(arrival.data_ptr()), self._stream()))
        failed = (arrival < 0).any(1)
        makespan = torch.where(failed, -1, arrival.max(1).values).to(torch.int32)
        soc = torch.where(failed, -1, arrival.sum(1)).to(torch.int32)
        return actions, arrival, makespan, soc

    def plan_orders(self, horizon: int = config.max_steps, orders: int = 8, seed: int = 0, env_offset: int = 0):
        """Prioritized planning over `orders` priority orders per environment (mapf_env_plan_prioritized_orders): order 0 is
        index order, order r >= 1 a Philox permutation of the agents drawn from (seed, env_offset + e, r), each planned as
        `plan` plans index order; an environment keeps its solved order of smallest sum of costs, ties to the smallest r.
        Returns (actions uint8[H,B,N], arrival int32[B,N], makespan int32[B], soc int32[B], order int32[B], rank
        uint8[B,N]) CUDA tensors on the current stream: the first four as `plan` returns them, for the winning order;
        order: the winning r, -1 where every order fails; rank: each agent's position in the winning order, 255 for absent
        agents and failed environments.  With orders=1 the first four equal `plan`'s.  The handle's state is not changed."""
        torch = _torch()
        B, N, H = self.num_envs, self.num_agents, int(horizon)
        actions = torch.empty((max(H, 1), B, N), dtype=torch.uint8, device=self.device)
        arrival = torch.empty((B, N), dtype=torch.int32, device=self.device)
        order = torch.empty(B, dtype=torch.int32, device=self.device)
        rank = torch.empty((B, N), dtype=torch.uint8, device=self.device)
        _native.check(self._lib.mapf_env_plan_prioritized_orders(
            self._h, H, int(orders), int(seed), int(env_offset), C.c_void_p(actions.data_ptr()),
            C.c_void_p(arrival.data_ptr()), C.c_void_p(order.data_ptr()), C.c_void_p(rank.data_ptr()), self._stream()))
        failed = (arrival < 0).any(1)
        makespan = torch.where(failed, -1, arrival.max(1).values).to(torch.int32)
        soc = torch.where(failed, -1, arrival.sum(1)).to(torch.int32)
        return actions, arrival, makespan, soc, order, rank

    def plan_lns(self, actions, arrival, iterations: int = 16, neighborhood: int = 8, seed: int = 0, env_offset: int = 0,
                 first_iteration: int = 0):
        """Improves a plan of the current state by large-neighbourhood search on the device (mapf_env_plan_lns): each
        iteration i re-plans a Philox-drawn group of `neighborhood` agents, by `plan`'s rules, against the other agents'
        paths, and keeps the new paths if their arrivals sum to strictly less.  `actions` uint8[H,B,N] and `arrival`
        int32[B,N] are CUDA tensors laid out as `plan` / `plan_orders` return them (or as this method returns them); they are
        copied, not changed.  Returns (actions, arrival, makespan, soc, accepted) CUDA tensors on the current stream: the
        improved plan as `plan` returns one, and accepted int32[B], the accepted iterations per environment, -1 where the
        input plan failed and -2 where it is not a valid plan of the current state (those environments are returned as they
        came).  The sum of costs never increases; calls split by `first_iteration` give one call's result.  The handle's state
        is not changed.  Defaults (DESIGN §8 (f)6, measured on a B200): after plan_orders(8) on 8192 x 32 @ 40, 16 iterations
        of 8 agents cost about 0.6x the orders call and reach the sum of costs of 16 orders in less time; on batches too small
        to fill the GPU (a few hundred environments) more orders are cheaper than more iterations."""
        torch = _torch()
        B, N = self.num_envs, self.num_agents
        assert actions.is_cuda and actions.dtype == torch.uint8 and actions.is_contiguous() and actions.dim() == 3
        assert tuple(actions.shape[1:]) == (B, N), "actions must be uint8 [H, B, N]"
        assert arrival.is_cuda and arrival.dtype == torch.int32 and tuple(arrival.shape) == (B, N), "arrival must be int32 [B, N]"
        H = int(actions.shape[0])
        actions, arrival = actions.clone(), arrival.contiguous().clone()
        accepted = torch.empty(B, dtype=torch.int32, device=self.device)
        _native.check(self._lib.mapf_env_plan_lns(
            self._h, H, int(iterations), int(neighborhood), int(seed), int(env_offset), int(first_iteration),
            C.c_void_p(actions.data_ptr()), C.c_void_p(arrival.data_ptr()), C.c_void_p(accepted.data_ptr()), self._stream()))
        failed = (arrival < 0).any(1)
        makespan = torch.where(failed, -1, arrival.max(1).values).to(torch.int32)
        soc = torch.where(failed, -1, arrival.sum(1)).to(torch.int32)
        return actions, arrival, makespan, soc, accepted

    def plan_repair(self, actions, arrival, iterations: int = 16, neighborhood: int = 8, seed: int = 0, env_offset: int = 0):
        """Repairs the failed environments of a plan on the device by collision-based large-neighbourhood search
        (mapf_env_plan_repair, MAPF-LNS2): an environment whose arrival row is -1 is planned again in index order with vertex
        collisions allowed but minimised, then up to `iterations` times a group of `neighborhood` agents (those with a
        collision first, in Philox order) is re-planned against the others and kept if the collision count drops, until no
        collision is left.  `actions` uint8[H,B,N] and `arrival` int32[B,N] are CUDA tensors laid out as `plan` /
        `plan_orders` / `plan_lns` return them; they are copied, not changed.  Returns (actions, arrival, makespan, soc,
        collisions) CUDA tensors on the current stream: the plan as `plan` returns one, and collisions int32[B]: 0 where the
        environment was repaired (a collision-free plan, valid input for `plan_lns`), G > 0 where G collisions were left
        (written as a failed plan), -1 where some agent has no path within H even with collisions, and -2 where the input was
        not a failed plan (returned as it came).  Where `plan` solves an environment, repairing its row of -1 gives `plan`'s
        plan.  The handle's state is not changed.  Defaults (DESIGN §8 (f)7, measured on a B200): 16 iterations of 8
        agents; after plan() on 8192 x 32 @ 40 they repair 1125 of 1141 failed environments in 82 ms, the solved fraction of
        plan_orders(32) in under a quarter of its time.  Environments left unrepaired run every iteration and set the call's
        time, so more iterations cost time almost linearly and repaired few more there."""
        torch = _torch()
        B, N = self.num_envs, self.num_agents
        assert actions.is_cuda and actions.dtype == torch.uint8 and actions.is_contiguous() and actions.dim() == 3
        assert tuple(actions.shape[1:]) == (B, N), "actions must be uint8 [H, B, N]"
        assert arrival.is_cuda and arrival.dtype == torch.int32 and tuple(arrival.shape) == (B, N), "arrival must be int32 [B, N]"
        H = int(actions.shape[0])
        actions, arrival = actions.clone(), arrival.contiguous().clone()
        collisions = torch.empty(B, dtype=torch.int32, device=self.device)
        _native.check(self._lib.mapf_env_plan_repair(
            self._h, H, int(iterations), int(neighborhood), int(seed), int(env_offset), C.c_void_p(actions.data_ptr()),
            C.c_void_p(arrival.data_ptr()), C.c_void_p(collisions.data_ptr()), self._stream()))
        failed = (arrival < 0).any(1)
        makespan = torch.where(failed, -1, arrival.max(1).values).to(torch.int32)
        soc = torch.where(failed, -1, arrival.sum(1)).to(torch.int32)
        return actions, arrival, makespan, soc, collisions

    def set_autoreset(self, max_steps: int = config.max_steps, seed: int = 0, env_offset: int = 0, stride: Optional[int] = None,
                      density: Optional[float] = None):
        """Episode handling inside `rollout` (worker.py:390,422-428): a step that finds its environment finished (done, or
        steps >= max_steps) re-generates the slot on the device instead of moving anybody -- the slot's n-th new instance
        is Philox stream (seed, env_offset + n * stride + e), what `reset(mask={e}, seed, env_offset + n * stride)` draws
        -- and emits the new episode's first observation with rewards 0 (code 5), done 0, steps 0.  `stride` = number of
        environments of the whole job (default: this batch).  max_steps = 0 switches it off."""
        dens = -1.0 if density is None else float(density)
        _native.check(self._lib.mapf_env_set_autoreset(self._h, int(max_steps), C.c_uint64(seed), C.c_uint64(env_offset),
                                                      C.c_uint64(stride if stride is not None else self.num_envs),
                                                      C.c_float(dens), self._stream()))

    def episode_counts(self):
        """int32[B] CUDA tensor: instances generated for each slot by the episode handling since set_autoreset."""
        torch = _torch()
        out = torch.empty((self.num_envs,), dtype=torch.int32, device=self.device)
        _native.check(self._lib.mapf_env_episode_counts(self._h, C.c_void_p(out.data_ptr()), self._stream()))
        return out

    def set_checks(self, check_unique: bool = True):
        """Post-step uniqueness check of the agents' cells (environment.py:424-428) in every step; a violation raises
        RuntimeError('unique') from check()."""
        _native.check(self._lib.mapf_env_set_checks(self._h, int(bool(check_unique))))

    def rollout_plan(self, num_steps: int, action_slots: int, obs_slots: int, out_slots: int, chains: int = 0):
        """-> (chains, envs_per_chain, graph_period) mapf_env_rollout would use (graph_period 0 = direct launches)."""
        out = [C.c_int32() for _ in range(3)]
        _native.check(self._lib.mapf_env_rollout_plan(self._h, int(num_steps), int(action_slots), int(obs_slots), int(out_slots),
                                                     int(chains), *[C.byref(o) for o in out]))
        return tuple(o.value for o in out)

    def observe(self, out_obs=None, obs_rows=None, out_bits=None):
        """-> (obs uint8[B,N,6,9,9], pos uint8[B,N,2])   (environment.py:433-467); `obs_rows` and `out_bits` (packed
        observations, returned in the observation's place) as in step()."""
        torch = _torch()
        B, N = self.num_envs, self.num_agents
        if out_bits is not None:
            assert out_obs is None, "out_bits replaces out_obs"
            pos = torch.empty((B, N, 2), dtype=torch.uint8, device=self.device)
            _native.check(self._lib.mapf_env_observe_packed(self._h, C.c_void_p(out_bits.data_ptr()),
                                                            self._bits_rows(out_bits, obs_rows), C.c_void_p(pos.data_ptr()),
                                                            self._stream()))
            return out_bits, pos
        obs = out_obs if out_obs is not None else torch.empty((B, N, *self.OBS_SHAPE), dtype=torch.uint8, device=self.device)
        pos = torch.empty((B, N, 2), dtype=torch.uint8, device=self.device)
        if obs_rows is not None:
            assert out_obs is not None and obs_rows.dtype == torch.int64 and obs_rows.is_cuda and obs_rows.numel() == B
            _native.check(self._lib.mapf_env_observe_rows(self._h, C.c_void_p(obs.data_ptr()), C.c_void_p(obs_rows.data_ptr()),
                                                          C.c_void_p(pos.data_ptr()), self._stream()))
            return obs, pos
        _native.check(self._lib.mapf_env_observe(self._h, C.c_void_p(obs.data_ptr()), C.c_void_p(pos.data_ptr()),
                                                 self._stream()))
        return obs, pos

    def comm_mask(self, max_comm_agents: int = config.max_comm_agents, out=None, out_bits=None, rows=None):
        """-> uint8[B,N,N] communication mask of Network.step (model.py:196-208) for the current positions:
        in each other's field of view AND among the `max_comm_agents` nearest (self included; ties -> lower id).
        `out_bits` (uint8 CUDA tensor [rows,N,ceil(N/8)]): the same launch also writes the mask as packed rows
        (`mapf_rl_b200.packed`), at row rows[e] (int64 CUDA tensor [B]) or row e; the dense mask is still returned."""
        torch = _torch()
        B, N = self.num_envs, self.num_agents
        m = out if out is not None else torch.empty((B, N, N), dtype=torch.uint8, device=self.device)
        assert m.is_contiguous() and m.dtype == torch.uint8 and m.numel() == B * N * N
        if out_bits is not None:
            rows_ptr = self._bits_rows(out_bits, rows, row_bytes=(N + 7) // 8)
            _native.check(self._lib.mapf_env_comm_mask_packed(self._h, int(max_comm_agents), C.c_void_p(m.data_ptr()),
                                                              C.c_void_p(out_bits.data_ptr()), rows_ptr, self._stream()))
            return m
        _native.check(self._lib.mapf_env_comm_mask(self._h, int(max_comm_agents), C.c_void_p(m.data_ptr()), self._stream()))
        return m

    def _host_buffers(self, want_obs: bool):
        """Page-locked host endpoints of step_host, allocated once and reused (DMA straight into them)."""
        torch = _torch()
        B, N = self.num_envs, self.num_agents
        hb = getattr(self, "_hb", None)
        if hb is None:
            # codes | steps | done of step_host_codes in ONE page-locked block, laid out like the library's device staging
            # (codes u8[B*N], pad to 16, steps i32[B], done u8[B]): the DMA form copies it back in one piece
            off_steps = (B * N + 15) & ~15
            off_done = off_steps + 4 * B
            block = torch.empty((off_done + B,), dtype=torch.uint8, pin_memory=True)
            hb = dict(actions=torch.empty((B, N), dtype=torch.uint8, pin_memory=True),
                      rewards=torch.empty((B, N), dtype=torch.float32, pin_memory=True),
                      codes=block[:B * N].view(B, N),
                      cdone=block[off_done:off_done + B],
                      csteps=block[off_steps:off_done].view(torch.int32),
                      done=torch.empty((B,), dtype=torch.uint8, pin_memory=True),
                      steps=torch.empty((B,), dtype=torch.int32, pin_memory=True))
            hb["_block"] = block
            hb.update({k + "_np": v.numpy() for k, v in list(hb.items()) if not k.startswith("_")})
            hb["ptrs"] = tuple(C.c_void_p(hb[k].data_ptr()) for k in ("actions", "rewards", "done", "steps"))
            hb["codes_ptrs"] = tuple(C.c_void_p(hb[k].data_ptr()) for k in ("codes", "cdone", "csteps"))
            self._hb = hb
        if want_obs and "obs" not in hb:
            hb["obs"] = torch.empty((B, N, *self.OBS_SHAPE), dtype=torch.uint8, pin_memory=True)
            hb["obs_np"] = hb["obs"].numpy()
        return hb

    @property
    def host_actions(self) -> np.ndarray:
        """uint8[B,N] page-locked action buffer of step_host; fill it in place and pass it to step_host to skip
        the staging copy."""
        return self._host_buffers(False)["actions_np"]

    def step_host(self, actions: np.ndarray, want_obs: bool = False, device_obs=None):
        """Host-buffer step through mapf_env_step_host: numpy (or a page-locked uint8 torch CPU tensor) in, numpy out,
        synchronous.
        Returns (obs | None, rewards, done, steps) as numpy VIEWS of page-locked buffers owned by this object:
        they are overwritten by the next step_host call (copy them to keep them)."""
        B, N = self.num_envs, self.num_agents
        hb = self._host_buffers(want_obs)
        pa, pr, pd, ps = hb["ptrs"]
        torch = _torch()
        pa = self._host_actions_ptr(actions, hb, pa)
        _native.check(self._lib.mapf_env_step_host(
            self._h, pa, hb["obs"].data_ptr() if want_obs else None, pr, pd, ps,
            C.c_void_p(device_obs.data_ptr()) if device_obs is not None else None, self._stream()))
        return (hb["obs_np"] if want_obs else None), hb["rewards_np"], hb["done_np"], hb["steps_np"]

    def _host_actions_ptr(self, actions, hb, default_ptr):
        """Pointer handed to the library for `actions`: a uint8 CPU tensor / the handle's own page-locked buffer is passed
        in place (the library checks on every call whether it is page-locked and stages it otherwise); anything else is
        copied into the handle's page-locked buffer first."""
        torch = _torch()
        B, N = self.num_envs, self.num_agents
        if isinstance(actions, torch.Tensor):
            assert (actions.device.type == "cpu" and actions.dtype == torch.uint8 and actions.is_contiguous()
                    and tuple(actions.shape) == (B, N)), "actions number"
            return C.c_void_p(actions.data_ptr())
        if actions is not hb["actions_np"]:   # the caller may fill env.host_actions in place instead
            a = np.asarray(actions)
            assert a.shape == (B, N), "actions number"
            np.copyto(hb["actions_np"], a, casting="unsafe")
        return default_ptr

    def step_host_codes(self, actions, device_obs):
        """Throughput form of the host-buffer step (mapf_env_step_host_codes): reward CODES instead of fp32 rewards, one
        fused kernel that publishes codes / done / steps straight into page-locked host memory; returns as soon as those
        are final, while the observation (device tensor `device_obs`, required) is still being written on the current
        stream.  Returns (codes uint8[B,N], done uint8[B], steps int32[B]) numpy VIEWS of page-locked buffers owned by this
        object (overwritten by the next call); rewards = reward_table[codes], see `reward_table`."""
        hb = getattr(self, "_hb", None) or self._host_buffers(False)
        pc, pd, ps = hb["codes_ptrs"]
        fast = hb.get("_fast")
        if fast is None:
            torch = _torch()
            fast = hb["_fast"] = (self._lib.mapf_env_step_host_codes, torch.Tensor, torch.cuda.current_stream)
        fn, tensor_t, cur = fast
        if type(actions) is tensor_t and actions.dtype is hb["actions"].dtype and actions.device.type == "cpu":
            # hot path of an actor that rotates over its own uint8 CPU tensors: shape / contiguity are checked once per buffer
            key = actions.data_ptr()
            seen = hb.setdefault("_seen", set())
            if key not in seen:
                assert actions.is_contiguous() and tuple(actions.shape) == (self.num_envs, self.num_agents), "actions number"
                if len(seen) > 256:
                    seen.clear()
                seen.add(key)
            pa = key
        else:
            pa = self._host_actions_ptr(actions, hb, hb["ptrs"][0])
        _native.check(fn(self._h, pa, pc, pd, ps, device_obs.data_ptr(), cur(self.device).cuda_stream))
        return hb["codes_np"], hb["cdone_np"], hb["csteps_np"]

    @property
    def reward_table(self) -> np.ndarray:
        """float32[6]: reward of each reward code (config.REWARD_ORDER, then 0 for a reset step)."""
        return np.asarray([float(self.reward_fn[k]) for k in config.REWARD_ORDER] + [0.0], dtype=np.float32)

    def check(self):
        """Synchronous: raise if a kernel latched an error (bad action -> AssertionError like the reference)."""
        _native.check(self._lib.mapf_env_status(self._h, self._stream()))

    # -- attributes (device tensors) -----------------------------------------------------------
    def _get_state(self, want):
        torch = _torch()
        B, N, L = self.num_envs, self.num_agents, self.map_length
        out = {}
        shapes = dict(map=((B, L, L), torch.uint8), pos=((B, N, 2), torch.uint8), goals=((B, N, 2), torch.uint8),
                      steps=((B,), torch.int32), navi=((B, N, 4, L, L), torch.uint8))
        ptrs = []
        for k in ("map", "pos", "goals", "steps", "navi"):
            if k in want:
                out[k] = torch.empty(shapes[k][0], dtype=shapes[k][1], device=self.device)
                ptrs.append(C.c_void_p(out[k].data_ptr()))
            else:
                ptrs.append(None)
        _native.check(self._lib.mapf_env_get_state(self._h, *ptrs, self._stream()))
        return out

    @property
    def steps(self):
        return self._get_state({"steps"})["steps"]

    @property
    def agents_pos(self):
        return self._get_state({"pos"})["pos"]

    @property
    def goals_pos(self):
        return self._get_state({"goals"})["goals"]

    @property
    def map(self):
        return self._get_state({"map"})["map"]

    @property
    def navi_map(self):
        """uint8[B,N,4,L,L]: navi_map without the obs_radius padding (environment.py:253-276)."""
        return self._get_state({"navi"})["navi"]

    def set_state(self, agents_pos=None, steps=None):
        torch = _torch()
        p = s = None
        if agents_pos is not None and self.sized:   # rows of absent agents are ignored (they read back as 255)
            ns, ls = (x.cpu().numpy().astype(np.int64) for x in self.sizes)
            p = self._coords_sized(agents_pos, ns, ls)
        elif agents_pos is not None:
            p = self._coords_u8(agents_pos, (self.num_envs, self.num_agents, 2))
        if steps is not None:
            s = torch.as_tensor(steps, dtype=torch.int32).to(self.device).contiguous()
        _native.check(self._lib.mapf_env_set_state(self._h, C.c_void_p(p.data_ptr()) if p is not None else None,
                                                   C.c_void_p(s.data_ptr()) if s is not None else None, self._stream()))
        self.check()   # synchronous; two agents on one cell -> RuntimeError('unique') (environment.py:424-428)

    def heuristic_distances(self, env_ids=None):
        """Recompute the BFS maps and return int32[n,N,L,L] distances (2147483647 = unreachable);
        equal to search.compute_heuristics (search.py:24-55) where finite."""
        torch = _torch()
        N, L = self.num_agents, self.map_length
        ids_ptr, n = None, self.num_envs
        if env_ids is not None:
            ids = torch.as_tensor(env_ids, dtype=torch.int32).to(self.device).contiguous()
            ids_ptr, n = C.c_void_p(ids.data_ptr()), int(ids.numel())
        dist = torch.empty((n, N, L, L), dtype=torch.int32, device=self.device)
        _native.check(self._lib.mapf_env_bfs_navi(self._h, ids_ptr, n, C.c_void_p(dist.data_ptr()), self._stream()))
        torch.cuda.current_stream(self.device).synchronize()
        return dist
