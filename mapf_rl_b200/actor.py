"""BatchedActor — the reference's rollout loop (Actor.run, worker.py:368-414) for B lockstep environments on
one GPU, with everything device-resident: the CUDA environment batch, a batched PyTorch Q-network, and
episode recording straight into a `ReplayStore` (the step kernel writes each observation at its final row
of the store; nothing is staged or copied).

Per step, as in the reference:
    q, hidden, comm_mask = model.step(obs, pos)            worker.py:378   (qnet.Network.step + comm-mask kernel)
    only agent 0 explores with probability epsilon         worker.py:380-382
    next_obs, r, done = env.step(actions)                  worker.py:385   (fused step + observe kernel)
    local_buffer.add(q[0], a[0], r[0], next_obs, hidden[0], comm_mask)     worker.py:388 / buffer.py:140-151
    episode end (done or env.steps >= max_steps):          worker.py:390-405
        initial priorities |TD| of LocalBuffer.finish      buffer.py:170-177 (actor_td kernel)
        GlobalBuffer.add: leaves = td ** alpha             worker.py:87-94   (sum-tree update kernel)
        env.reset                                          worker.py:422-428 (device generator + BFS)
With a `Curriculum` (sized environment batch), every reset draws each slot's (num_agents, map_length) from the
curriculum's current levels (worker.py:424-425) and finished episodes of the counted environments record their setting
and done flag in it (worker.py:73-82).  Absent agents' rows of the store are zeros.
Every environment owns one episode slot of the store while its episode runs; a finished episode is published
(priorities inserted, size / done recorded) and the environment takes the next free slot of the ring, whose
old leaves are zeroed first so a half-overwritten episode is never sampled.  The only host synchronisation
per step is the read of the B-byte "episode finished" mask.
With a compact store (`ReplayStore(compact=True)`) the step kernel and the comm-mask kernel write packed rows, the current
frames are unpacked from the store for the Q-network (mapf_obs_unpack), and one hidden vector is kept per transition; the
store then holds exactly what the dense store would.
With `present_only=True` the Q-network's encoder and input GRU run on present agents only (`present.py`): the present rows
are rebuilt at every episode start (agent counts change only at resets), the current frames come in that layout
(mapf_obs_unpack_present with a compact store, indexing obs_buf with a dense one), and the store receives what it receives
without.  The results equal the padded path's up to floating-point reordering, not bit for bit.
"""
from __future__ import annotations

from typing import Callable, Optional

import numpy as np

from . import config
from .batched import BatchedEnvironment
from .buffer import actor_td_errors
from .present import PresentRows
from .replay import ReplayStore


def _torch():
    import torch
    return torch


class BatchedActor:
    def __init__(self, env: BatchedEnvironment, net, store: ReplayStore, epsilon=0.1, seed: int = 0,
                 density: Optional[float] = None, max_steps: int = config.max_steps,
                 on_step: Optional[Callable] = None, on_episode: Optional[Callable] = None,
                 on_begin: Optional[Callable] = None, curriculum=None, curriculum_envs=None, present_only: bool = False):
        """curriculum: a `Curriculum` whose levels the resets draw from (needs `BatchedEnvironment(..., sized=True)`);
        curriculum_envs: the environments whose finished episodes it counts (default: all; the reference counts its
        low-epsilon actors, ids 10-15, only); present_only: run the network's encoder on present agents only (`net.step`
        takes `present=`)."""
        torch = _torch()
        assert curriculum is None or env.sized, "a curriculum needs a sized environment batch"
        self.curriculum = curriculum
        self._counted = np.ones(env.num_envs, dtype=bool)
        if curriculum_envs is not None:
            self._counted[:] = False
            self._counted[np.asarray(curriculum_envs, dtype=np.int64)] = True
        assert store.max_num_agents == env.num_agents, "the store is laid out for the batch's agent count"
        assert store.capacity >= 2 * env.num_envs, "capacity >= 2 * num_envs (a power of two): every env owns a slot while it runs"
        assert max_steps <= store.max_steps
        self.env, self.net, self.store = env, net, store
        self.B, self.N, self.dev = env.num_envs, env.num_agents, env.device
        self.max_steps, self.density, self.seed = int(max_steps), density, int(seed)
        self.epsilon = torch.as_tensor(epsilon, dtype=torch.float32, device=self.dev).expand(self.B).contiguous()
        self.gen = torch.Generator(device=self.dev)
        self.gen.manual_seed(self.seed)
        self.on_step, self.on_episode, self.on_begin = on_step, on_episode, on_begin
        S = store.max_steps
        self.q_buf = torch.zeros((self.B, S, 5), dtype=torch.float32, device=self.dev)      # LocalBuffer.q_buf rows 0..size-1
        self.slot = torch.zeros(self.B, dtype=torch.int64, device=self.dev)                  # episode slot of each env
        self.t = torch.zeros(self.B, dtype=torch.int64, device=self.dev)                     # == env.steps
        self._slot_host = np.zeros(self.B, dtype=np.int64)
        self._owned = set()
        self.episodes = 0
        self.transitions = 0
        self.resets = 0
        self._started = False
        self.present_only = bool(present_only)
        self.present = None

    # -- slots ---------------------------------------------------------------------------------------
    def _take_slots(self, count: int) -> np.ndarray:
        st = self.store
        out = []
        while len(out) < count:
            s = st.ptr
            st.ptr = (st.ptr + 1) % st.capacity
            if s in self._owned:
                continue                       # an episode still running there: never evict it
            out.append(s)
            self._owned.add(s)
        slots = np.asarray(out, dtype=np.int64)
        # evict: the old episodes of these slots must not be sampled while they are overwritten
        st.size -= int(st._size_host[slots].sum())
        st._size_host[slots] = 0
        S = st.max_steps
        leaves = (slots[:, None] * S + np.arange(S)[None, :]).reshape(-1)
        torch = _torch()
        st.priority_tree.update_device(torch.as_tensor(leaves, device=self.dev),
                                       torch.zeros(leaves.shape[0], dtype=torch.float64, device=self.dev))
        sl = torch.as_tensor(slots, device=self.dev)
        st.size_buf[sl] = 0
        st.done_buf[sl] = 0
        return slots

    def _rows(self):
        return self.slot * (self.store.max_steps + 1) + self.t     # observation / comm row of the current frame

    # -- episode start for the envs in `ids` (all on the first call) ------------------------------------
    def _begin(self, ids: np.ndarray, first: bool):
        torch = _torch()
        mask = torch.zeros(self.B, dtype=torch.uint8, device=self.dev)
        idt = torch.as_tensor(ids, device=self.dev)
        mask[idt] = 1
        self.resets += 1
        # fresh instances: slot e of reset number r draws global stream (seed, r * B + e)
        self.env.reset(mask=None if first else mask, seed=self.seed, env_offset=self.resets * self.B, density=self.density,
                       levels=self.curriculum.levels if self.curriculum is not None else None)
        # a generator that could not place its agents latches MAPF_ERRBIT_RESET and leaves the slot as it was: surface it
        # here instead of stepping stale positions on a new map (one 4-byte status read per batch of episode ends; the
        # Q-network forward between two steps is three orders of magnitude longer)
        self.env.check()
        slots = self._take_slots(len(ids))
        self._slot_host[ids] = slots
        self.slot[idt] = torch.as_tensor(slots, device=self.dev)
        counts = self.env.sizes[0] if self.env.sized else torch.full((self.B,), self.N, dtype=torch.uint8, device=self.dev)
        self.store.agents_buf[self.slot[idt]] = counts[idt]                     # num_agents of the slot's episode
        if self.present_only:
            self.present = PresentRows(counts, int(counts.sum(dtype=torch.int64).item()), self.N)
        self.t[idt] = 0
        # frame 0 of the new episodes (LocalBuffer.__init__: obs_buf[0] = init_obs, buffer.py:131); environments
        # in the middle of an episode rewrite the frame they already hold
        self.env.observe(**self.store.frame_out(), obs_rows=self._rows())
        if self.on_begin is not None:
            self.on_begin(self, ids)
        return mask

    # -- one lockstep step -----------------------------------------------------------------------------
    def step(self):
        torch = _torch()
        st, env, B = self.store, self.env, self.B
        S = st.max_steps
        reset_mask = None
        if not self._started:
            self._begin(np.arange(B), first=True)
            self.net.reset()
            self._started = True
        rows = self._rows()
        pr = self.present
        obs = st.current_frames(rows, pr)                                        # [B,N,6,9,9] or [M_pad,6,9,9]
        comm = st.record_comm(env, rows)                                         # model.py:196-208, -> comm_buf[size]
        if pr is not None:
            actions, q, hidden = self.net.step(obs, comm, reset_mask=self._pending_reset, present=pr)
        else:
            actions, q, hidden = self.net.step(obs, comm, reset_mask=self._pending_reset)
        self._pending_reset = None
        # only agent 0 explores (worker.py:380-382)
        explore = torch.rand(B, device=self.dev, generator=self.gen) < self.epsilon
        rnd = torch.randint(0, 5, (B,), device=self.dev, generator=self.gen)
        actions = actions.clone()
        actions[:, 0] = torch.where(explore, rnd, actions[:, 0])
        a8 = actions.to(torch.uint8)
        _, rewards, done = env.step(a8, **st.frame_out(), obs_rows=rows + 1)     # next_obs -> obs_buf[size + 1]
        # local_buffer.add(q_val[0], actions[0], r[0], next_obs, hidden[0], comm_mask)  (worker.py:388, buffer.py:140-151)
        leaf = self.slot * S + self.t
        st.act_buf[leaf] = a8[:, 0]
        st.rew_buf[leaf] = rewards[:, 0].to(torch.float16)
        st.write_hidden(leaf, hidden[:, 0])                                      # agent 0's vector
        self.q_buf[torch.arange(B, device=self.dev), self.t] = q[:, 0, :].float()
        self.t += 1
        self.transitions += B
        if self.on_step is not None:
            self.on_step(self, a8, rewards, done)
        # episode end: done or env.steps >= max_steps (worker.py:390)
        fin_dev = (done != 0) | (self.t >= self.max_steps)
        fin = fin_dev.cpu().numpy()                                              # the one host sync of the step
        ids = np.flatnonzero(fin)
        if ids.size:
            self._finish(ids)
            self._begin(ids, first=False)
            self._pending_reset = fin_dev                                        # model.reset() for those envs (worker.py:423)
        return rewards, done

    _pending_reset = None

    # -- LocalBuffer.finish + GlobalBuffer.add for the envs in `ids` -------------------------------------
    def _finish(self, ids: np.ndarray):
        torch = _torch()
        st = self.store
        S = st.max_steps
        idt = torch.as_tensor(ids, device=self.dev)
        slots, size = self.slot[idt], self.t[idt]
        done = self.env._done[idt] != 0
        st.close_comm(slots * (S + 1) + size, done)                             # comm_buf[size]
        # initial priorities (buffer.py:170-177) and their insertion (worker.py:87-94)
        leaves = (slots[:, None] * S + torch.arange(S, device=self.dev)[None, :])
        rew = st.rew_buf[leaves].float()
        act = st.act_buf[leaves]
        td = actor_td_errors(rew, self.q_buf[idt], act, size.to(torch.int32), capacity=S, device=self.dev,
                             forward_steps=st.forward_steps)
        st.priority_tree.update_device(leaves.reshape(-1), td.reshape(-1) ** st.alpha)
        st.done_buf[slots] = done.to(torch.uint8)
        st.size_buf[slots] = size.to(torch.int32)
        size_h = size.cpu().numpy()
        for s, n in zip(self._slot_host[ids], size_h):
            st._size_host[s] = int(n)
            self._owned.discard(int(s))
        st.size += int(size_h.sum())
        st.counter += int(size_h.sum())
        self.episodes += len(ids)
        if self.curriculum is not None:
            counted = ids[self._counted[ids]]
            if counted.size:
                n_e, l_e = (x.cpu().numpy() for x in self.env.sizes)
                self.curriculum.record(n_e[counted], l_e[counted], self.env._done[torch.as_tensor(counted, device=self.dev)].cpu().numpy() != 0)
        if self.on_episode is not None:
            self.on_episode(self, ids, self._slot_host[ids].copy(), size_h, done.cpu().numpy(), td)

    def run(self, steps: int):
        for _ in range(steps):
            self.step()
