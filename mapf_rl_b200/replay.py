"""ReplayStore — device-resident mirror of the storage and sampling half of the reference's `GlobalBuffer`
(worker.py:21-203, without Ray; the curriculum statistics are `curriculum.Curriculum`).

The buffers keep the reference's logical layout (worker.py:36-42) as CUDA tensors: episode slot g owns
observation / comm-mask rows g*(max_steps+1)+f and action / reward / hidden rows g*max_steps+t, and the
priority tree leaf of transition (g, t) is g*max_steps+t.  Observations are stored as the bool bytes the
step kernel emits, so a batched actor can point `BatchedEnvironment.step(out_obs=...)` straight at rows
of `obs_buf`.  `sample_batch` is two launches: the sum-tree descent (mapf_per_sample) and the window
gather with bool->fp16 conversion (mapf_replay_gather); `update_priorities` is the fused stale-mask +
tree update.  Return values follow the reference's tuple (worker.py:168-182) with CUDA tensors in
place of CPU ones.

`compact=True` keeps the same logical store in about a twelfth of the memory at 32 agents (DESIGN.md §3): observations
and comm masks as packed bits (`obs_bits`, `comm_bits`, formats in `mapf_rl_b200.packed`) and one hidden vector per
transition (`hid_buf` [max_steps*capacity, latent]; the reference writes agent 0's vector into every agent's row,
buffer.py:148).  `gather` / `sample_batch` return exactly what the dense store returns for the same contents.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional

import numpy as np

from . import _native, config, packed
from .present import PresentRows, unpack_obs_present
from .buffer import SumTree


def _torch():
    import torch
    return torch


class ReplayStore:
    def __init__(self, capacity: int, alpha=config.prioritized_replay_alpha, beta=config.prioritized_replay_beta,
                 max_num_agents: int = config.max_num_agents, device=None, max_steps: int = config.max_steps,
                 bt_steps: int = config.bt_steps, forward_steps: int = config.forward_steps,
                 latent_dim: int = config.latent_dim, compact: bool = False):
        torch = _torch()
        if not torch.cuda.is_available():
            raise RuntimeError("mapf_rl_b200 needs a CUDA device: the replay kernels have no CPU fallback")
        self._lib = _native.lib()
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.capacity, self.alpha, self.beta = int(capacity), alpha, beta
        self.max_num_agents, self.max_steps = int(max_num_agents), int(max_steps)
        self.bt_steps, self.forward_steps, self.latent_dim = int(bt_steps), int(forward_steps), int(latent_dim)
        self.size = 0       # stored transitions (worker.py:25)
        self.ptr = 0        # next episode slot (worker.py:26)
        self.counter = 0
        self.priority_tree = SumTree(self.capacity * self.max_steps, device=self.device)   # worker.py:27
        n, S, dev = self.max_num_agents, self.max_steps, self.device
        z = lambda shape, dt: torch.zeros(shape, dtype=dt, device=dev)
        self.compact = bool(compact)
        if self.compact:
            self.obs_bits = z(((S + 1) * capacity, n, packed.OBS_BYTES), torch.uint8)
            self.comm_bits = z(((S + 1) * capacity, n, packed.comm_bytes(n)), torch.uint8)
            self.hid_buf = z((S * capacity, self.latent_dim), torch.float16)
        else:
            self.obs_buf = z(((S + 1) * capacity, n, *config.obs_shape), torch.uint8)      # worker.py:36
            self.hid_buf = z((S * capacity, n, self.latent_dim), torch.float16)            # worker.py:39
            self.comm_mask = z(((S + 1) * capacity, n, n), torch.uint8)                    # worker.py:42
        self.act_buf = z((S * capacity,), torch.uint8)                                     # worker.py:37
        self.rew_buf = z((S * capacity,), torch.float16)                                   # worker.py:38
        self.done_buf = z((capacity,), torch.uint8)                                        # worker.py:40
        self.size_buf = z((capacity,), torch.int32)                                        # worker.py:41
        # agents of each slot's episode (the tuple's num_agents, worker.py:72); N until written, so an unannotated slot reads as
        # padded.  gather(present=True) lays its rows out by it.
        self.agents_buf = torch.full((capacity,), n, dtype=torch.uint8, device=dev)
        self._size_host = np.zeros(capacity, dtype=np.int64)
        self._err = z((1,), torch.int32)

    def __len__(self):
        return self.size

    @staticmethod
    def bytes_per_transition(num_agents: int, latent_dim: int = config.latent_dim, compact: bool = False) -> int:
        """Device bytes one stored transition takes: its observation and comm-mask frame, hidden state, action and reward
        (without the extra frame per episode slot, the per-slot done / size and the sum tree)."""
        n = int(num_agents)
        if compact:
            frame = n * packed.OBS_BYTES + n * packed.comm_bytes(n) + 2 * int(latent_dim)
        else:
            frame = n * packed.OBS_ELEMS + n * n + 2 * n * int(latent_dim)
        return frame + 1 + 2

    @property
    def nbytes(self) -> int:
        """Device bytes of the store's buffers (without the sum tree, which is the same for both layouts)."""
        bufs = ((self.obs_bits, self.comm_bits) if self.compact else (self.obs_buf, self.comm_mask)) + (
            self.hid_buf, self.act_buf, self.rew_buf, self.done_buf, self.size_buf, self.agents_buf)
        return sum(b.numel() * b.element_size() for b in bufs)

    def _stream(self):
        return C.c_void_p(_torch().cuda.current_stream(self.device).cuda_stream)

    # -- GlobalBuffer.add (worker.py:68-104) ------------------------------------------------------
    def add(self, buffer_list: List):
        """buffer_list: tuples as returned by LocalBuffer.finish — actor_id 0, num_agents 1, map_len 2, obs_buf 3,
        act_buf 4, rew_buf 5, hid_buf 6, td_errors 7, done 8, size 9, comm_mask 10 (worker.py:72).
        A compact store packs observations and comm masks on the host (agents >= num_agents get zero rows) and keeps one
        hidden vector per transition: it raises ValueError if a transition's hidden rows differ, which the reference never
        writes (buffer.py:148).  num_agents goes to `agents_buf`; it raises ValueError outside 1..max_num_agents."""
        torch = _torch()
        S = self.max_steps
        dev = self.device
        for b in buffer_list:
            if not 1 <= int(b[1]) <= self.max_num_agents:
                raise ValueError(f"num_agents {int(b[1])} outside 1..{self.max_num_agents}")

        def up(x, dt):
            return torch.as_tensor(np.ascontiguousarray(x)).to(device=dev, dtype=dt, non_blocking=True)

        if self.compact:   # check every tuple before anything is written
            hids = [packed.single_hidden(np.asarray(b[6], dtype=np.float16)[:int(b[9])]) for b in buffer_list]
        for k, buffer in enumerate(buffer_list):
            n, size = int(buffer[1]), int(buffer[9])
            idxes = np.arange(self.ptr * S, (self.ptr + 1) * S, dtype=np.int64)            # worker.py:88
            start_idx = self.ptr * S
            self.size -= int(self._size_host[self.ptr])
            self.size += size
            self.counter += size
            self.priority_tree.batch_update(idxes, np.asarray(buffer[7], dtype=np.float64) ** self.alpha)   # worker.py:94
            row0 = start_idx + self.ptr                                                    # = ptr * (S + 1)
            if self.compact:
                N = self.max_num_agents
                obs = np.zeros((size + 1, N, *config.obs_shape), dtype=np.uint8)
                obs[:, :n] = np.asarray(buffer[3])[:size + 1]
                comm = np.zeros((size + 1, N, N), dtype=np.uint8)
                comm[:, :n, :n] = np.asarray(buffer[10])[:size + 1]
                self.obs_bits[row0:row0 + size + 1] = up(packed.pack_obs(obs), torch.uint8)
                self.comm_bits[row0:row0 + size + 1] = up(packed.pack_comm(comm), torch.uint8)
                self.hid_buf[start_idx:start_idx + size] = up(hids[k], torch.float16)
            else:
                self.obs_buf[row0:row0 + size + 1, :n] = up(buffer[3], torch.uint8)        # worker.py:96
                self.hid_buf[start_idx:start_idx + size, :n] = up(np.asarray(buffer[6], dtype=np.float16), torch.float16)
                self.comm_mask[row0:row0 + size + 1, :n, :n] = up(buffer[10], torch.uint8)  # worker.py:102
            self.act_buf[start_idx:start_idx + size] = up(buffer[4], torch.uint8)
            self.rew_buf[start_idx:start_idx + size] = up(np.asarray(buffer[5], dtype=np.float16), torch.float16)
            self.done_buf[self.ptr] = int(bool(buffer[8]))
            self.size_buf[self.ptr] = size
            self.agents_buf[self.ptr] = n
            self._size_host[self.ptr] = size
            self.ptr = (self.ptr + 1) % self.capacity

    # -- direct-write path of a batched actor -------------------------------------------------------
    def obs_rows(self, slot: int, first_frame: int, count: int):
        """View of `count` consecutive observation frames of episode slot `slot` — the tensor a batched actor
        passes as `out_obs` (`out_bits`: packed rows of a compact store) so the step kernel writes into the replay store
        with no copy."""
        row0 = slot * (self.max_steps + 1) + first_frame
        return (self.obs_bits if self.compact else self.obs_buf)[row0:row0 + count]

    def frame_out(self) -> dict:
        """The keyword argument that makes `BatchedEnvironment.step` / `observe` (with `obs_rows`) write observations into
        the store's frame rows: `out_obs`, or `out_bits` (packed rows) for a compact store."""
        return dict(out_bits=self.obs_bits) if self.compact else dict(out_obs=self.obs_buf)

    def current_frames(self, rows, present: Optional[PresentRows] = None):
        """The observation frames at `rows` (int64 CUDA tensor [B], frame e of environment e) for the Q-network: uint8
        [B, N, 6, 9, 9], or [M_pad, 6, 9, 9] in the present-agent rows of `present`."""
        if self.compact:
            return packed.unpack_obs(self.obs_bits, rows) if present is None else unpack_obs_present(self.obs_bits, rows, present)
        obs = self.obs_buf.index_select(0, rows)
        return obs if present is None else present.select(obs.flatten(0, 1))

    def record_comm(self, env, rows):
        """The comm mask of `env`'s current positions (model.py:196-208) -> uint8 CUDA tensor [B, N, N], also stored at frame
        `rows` (comm_buf[size] = comm_mask, buffer.py:149)."""
        if self.compact:
            return env.comm_mask(out_bits=self.comm_bits, rows=rows)     # the packed rows in the same launch
        comm = env.comm_mask()
        self.comm_mask.index_copy_(0, rows, comm)
        return comm

    def close_comm(self, last_rows, done):
        """comm_buf[size] of finished episodes (`last_rows`, their frame after the last step): the mask of the last step, which
        `record_comm` stored at the row before, when the episode was cut at max_steps (worker.py:399-401; the reference re-runs
        the model on the PREVIOUS observation there), zeros when it ended by `done` (buffer.py:124,155-156)."""
        torch = _torch()
        buf = self.comm_bits if self.compact else self.comm_mask
        prev = buf[last_rows - 1]
        buf[last_rows] = torch.where(done[:, None, None], torch.zeros_like(prev), prev)

    def write_hidden(self, leaf, hidden):
        """Agent 0's hidden vector (`hidden` [B, latent]) of the transitions at `leaf`: once in a compact store, in each agent's
        row of a dense one, as the reference broadcasts it (buffer.py:148, SURVEY q8)."""
        h = hidden.to(_torch().float16)
        self.hid_buf[leaf] = h if self.compact else h[:, None, :].expand(-1, self.max_num_agents, -1)

    # -- GlobalBuffer.sample_batch (worker.py:106-184) ------------------------------------------------
    def _view(self):
        if self.compact:
            return _native.ReplayViewCompact(self.obs_bits.data_ptr(), self.comm_bits.data_ptr(), self.hid_buf.data_ptr(),
                                             self.act_buf.data_ptr(), self.rew_buf.data_ptr(), self.done_buf.data_ptr(),
                                             self.size_buf.data_ptr(), self.max_num_agents, self.max_steps, self.bt_steps,
                                             self.forward_steps, self.latent_dim)
        return _native.ReplayView(self.obs_buf.data_ptr(), self.comm_mask.data_ptr(), self.hid_buf.data_ptr(),
                                  self.act_buf.data_ptr(), self.rew_buf.data_ptr(), self.done_buf.data_ptr(),
                                  self.size_buf.data_ptr(), self.max_num_agents, self.max_steps, self.bt_steps,
                                  self.forward_steps, self.latent_dim)

    def gather(self, idxes, present: bool = False):
        """Window gather for the given leaf indices (int64 CUDA tensor [B]) -> dict of CUDA tensors.
        present=True: observations [M_pad, W, 6, 9, 9] and hidden [M_pad, latent] in present-agent rows (`present.py`, one
        row per agent a < agents_buf[slot] of each sample), under "present" the `PresentRows` of the batch; comm_mask and the
        scalars as without.  Sizing the output reads M on the host (one small device-to-host copy)."""
        torch = _torch()
        idx = torch.as_tensor(idxes, dtype=torch.int64).to(self.device).contiguous()
        if present:
            return self._gather_present(idx)
        B, n, W = int(idx.numel()), self.max_num_agents, self.bt_steps + self.forward_steps
        out, batch = self._outputs(B, (B, W, n), B * n)
        gather = self._lib.mapf_replay_gather_compact if self.compact else self._lib.mapf_replay_gather
        _native.check(gather(C.byref(self._view()), C.c_void_p(idx.data_ptr()), B, C.byref(batch),
                             C.c_void_p(self._err.data_ptr()), self._stream()))
        return out

    def _outputs(self, B: int, obs_rows, hidden_rows: int):
        """Uninitialised outputs of a gather of B samples -> (dict, its `ReplayBatch`); obs is [*obs_rows, 6, 9, 9] and hidden
        [hidden_rows, latent], in padded or present-agent rows."""
        torch = _torch()
        n, W = self.max_num_agents, self.bt_steps + self.forward_steps
        e = lambda shape, dt: torch.empty(shape, dtype=dt, device=self.device)
        out = dict(obs=e((*obs_rows, *config.obs_shape), torch.float16), comm_mask=e((B, W, n, n), torch.uint8),
                   hidden=e((hidden_rows, self.latent_dim), torch.float16), action=e((B,), torch.int64),
                   reward=e((B,), torch.float16), done=e((B,), torch.float16), steps=e((B,), torch.float16),
                   bt_steps=e((B,), torch.int64))
        batch = _native.ReplayBatch(*[out[k].data_ptr() for k in ("obs", "comm_mask", "hidden", "action", "reward", "done",
                                                                   "steps", "bt_steps")])
        return out, batch

    def _gather_present(self, idx):
        torch = _torch()
        # an entry above N reads as N, as mapf_replay_gather_present reads it
        counts = self.agents_buf[idx // self.max_steps].clamp(max=self.max_num_agents)
        pr = PresentRows(counts, int(counts.sum(dtype=torch.int64).item()), self.max_num_agents)
        W = self.bt_steps + self.forward_steps
        if not self.compact:   # the padded gather, indexed: also the reference the kernel is tested against
            out = self.gather(idx)
            out["obs"] = pr.select(out["obs"].transpose(1, 2).reshape(pr.B * pr.N, W, *config.obs_shape))
            out["hidden"] = pr.select(out["hidden"])
            out["present"] = pr
            return out
        out, batch = self._outputs(pr.B, (pr.M_pad, W), pr.M_pad)
        _native.check(self._lib.mapf_replay_gather_present(
            C.byref(self._view()), C.c_void_p(self.agents_buf.data_ptr()), C.c_void_p(idx.data_ptr()),
            C.c_void_p(pr.first.data_ptr()), pr.B, pr.M_pad, C.byref(batch), C.c_void_p(self._err.data_ptr()), self._stream()))
        out["present"] = pr
        return out

    def sample_batch(self, batch_size: int, uniforms=None, check: bool = True):
        """-> (obs f16[B,W,n,6,9,9], action i64[B,1], reward f16[B,1], done f16[B,1], steps f16[B,1], bt_steps i64[B],
        hidden f16[B*n,latent], comm_mask bool[B,W,n,n], idxes int64 numpy[B], weights f16[B,1], ptr) — the reference's
        tuple (worker.py:168-182) with CUDA tensors.  `uniforms` (optional, [B] in [0,1)) replaces the draw
        np.random.uniform makes inside SumTree.batch_sample (buffer.py:60)."""
        torch = _torch()
        if uniforms is None:
            uniforms = np.random.random_sample(batch_size)
        idx, prio, _ = self.priority_tree.sample_device(batch_size, uniforms)
        out = self.gather(idx)
        # importance sampling weights (worker.py:165-166), fp64 like numpy, then fp16 (:181)
        weights = (prio / prio.min()).pow(-self.beta).to(torch.float16).unsqueeze(1)
        idx_host = idx.cpu().numpy()
        if check:
            if int(self._err.item()) != 0:
                self._err.zero_()
                raise AssertionError("sampled transition lies beyond its episode (worker.py:120)")
        return (out["obs"], out["action"].unsqueeze(1), out["reward"].unsqueeze(1), out["done"].unsqueeze(1),
                out["steps"].unsqueeze(1), out["bt_steps"], out["hidden"], out["comm_mask"].bool(), idx_host, weights,
                self.ptr)

    # -- GlobalBuffer.update_priorities (worker.py:186-203) --------------------------------------------
    def update_priorities(self, idxes: np.ndarray, priorities: np.ndarray, old_ptr: int):
        idxes = np.asarray(idxes)
        priorities = np.asarray(priorities)
        S = self.max_steps
        if self.ptr > old_ptr:      # discard the slots overwritten since sampling: [old_ptr, ptr)
            mask = (idxes < old_ptr * S) | (idxes >= self.ptr * S)
            idxes, priorities = idxes[mask], priorities[mask]
        elif self.ptr < old_ptr:    # [0, ptr) and [old_ptr, capacity)
            mask = (idxes < old_ptr * S) & (idxes >= self.ptr * S)
            idxes, priorities = idxes[mask], priorities[mask]
        # numpy evaluates priorities**alpha in the dtype the learner sent (fp16 in the reference, SURVEY a15)
        self.priority_tree.batch_update(np.array(idxes, dtype=np.int64), priorities ** self.alpha)

    def update_priorities_device(self, q_online, q_target_next, action, reward, done, steps, idxes, old_ptr: int,
                                 gamma: float = 0.99, q_online_next=None):
        """Learner tail on the device: TD error, priority, stale mask and tree update in one launch
        (SumTree.td_update).  Returns (td, priority) CUDA tensors."""
        return self.priority_tree.td_update(q_online, q_target_next, action, reward, done, steps, idxes, old_ptr=old_ptr,
                                            ptr=self.ptr, slot_steps=self.max_steps, gamma=gamma, alpha=self.alpha,
                                            q_online_next=q_online_next)

    def ready(self):  # worker.py:228-232
        return len(self) >= config.learning_starts
