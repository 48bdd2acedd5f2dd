"""Mirror of the reference's replay primitives (buffer.py:16-179) over device memory.

`SumTree` keeps the fp64 array heap in HBM (it is 8 MiB at the reference's 2^19 leaves and stays in
L2); `batch_sample` / `batch_update` / `td_update` are single launches of the kernels in
csrc/mapf_per_kernels.cu through the C ABI.  `LocalBuffer` keeps the reference's per-episode numpy
storage (it is an API mirror, the storage itself is a "next" row of the scope table) and computes the
initial priorities of `finish()` on the device.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _native, config


def _torch():
    import torch
    return torch


class _CudaArrayView:
    def __init__(self, ptr, n, owner):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<f8", "data": (ptr, False), "version": 2}
        self._owner = owner


class SumTree:
    """buffer.SumTree (buffer.py:16-105).  `tree` is a float64 CUDA tensor aliasing the device heap."""

    def __init__(self, capacity, device=None):
        torch = _torch()
        if not torch.cuda.is_available():
            raise RuntimeError("mapf_rl_b200 needs a CUDA device: the sum-tree kernels have no CPU fallback")
        layer = 1
        while 2 ** (layer - 1) < capacity:
            layer += 1
        assert 2 ** (layer - 1) == capacity, 'buffer size only support power of 2 size'
        self.layer = layer
        self.capacity = capacity
        self.size = 0
        self._lib = _native.lib()
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        h = C.c_void_p()
        _native.check(self._lib.mapf_per_create(int(capacity), self.device.index, C.byref(h)))
        self._h = h
        ptr = self._lib.mapf_per_tree_ptr(h)
        with torch.cuda.device(self.device):
            self.tree = torch.as_tensor(_CudaArrayView(ptr, 2 ** layer - 1, self), device=self.device)

    def close(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            self.tree = None
            self._lib.mapf_per_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return C.c_void_p(_torch().cuda.current_stream(self.device).cuda_stream)

    def sum(self):  # buffer.py:29-31
        return float(self.tree[0].item())

    def __getitem__(self, idx: int):  # buffer.py:33-36
        assert 0 <= idx < self.capacity
        return float(self.tree[self.capacity - 1 + idx].item())

    # -- device-tensor API (fast path) ---------------------------------------------------------
    def sample_device(self, batch_size: int, uniforms=None, beta=None):
        """-> (idx int64[B], priority float64[B], is_weight float32[B] | None) CUDA tensors."""
        torch = _torch()
        if uniforms is None:
            uniforms = torch.rand(batch_size, dtype=torch.float64, device=self.device)
        u = torch.as_tensor(uniforms, dtype=torch.float64).to(self.device).contiguous()
        idx = torch.empty(batch_size, dtype=torch.int64, device=self.device)
        pr = torch.empty(batch_size, dtype=torch.float64, device=self.device)
        w = torch.empty(batch_size, dtype=torch.float32, device=self.device) if beta is not None else None
        _native.check(self._lib.mapf_per_sample(self._h, C.c_void_p(u.data_ptr()), batch_size, C.c_void_p(idx.data_ptr()),
                                                C.c_void_p(pr.data_ptr()), C.c_void_p(w.data_ptr()) if w is not None else None,
                                                float(beta or 0.0), self._stream()))
        return idx, pr, w

    def update_device(self, idx, prio):
        """leaf[idx[k]] = prio[k] (last duplicate wins) + ancestor refresh; CUDA tensors int64 / float64."""
        torch = _torch()
        idx = torch.as_tensor(idx, dtype=torch.int64).to(self.device).contiguous()
        prio = torch.as_tensor(prio, dtype=torch.float64).to(self.device).contiguous()
        assert idx.shape == prio.shape
        # asynchronous on the current stream (device tensors are released stream-ordered by torch's allocator)
        _native.check(self._lib.mapf_per_update(self._h, C.c_void_p(idx.data_ptr()), C.c_void_p(prio.data_ptr()),
                                                int(idx.numel()), self._stream()))

    def td_update(self, q_online, q_target_next, action, reward, done, steps, idx, old_ptr=0, ptr=0,
                  slot_steps=config.max_steps, gamma=0.99, alpha=config.prioritized_replay_alpha, q_online_next=None):
        """Fused learner tail (worker.py:300-308 + 186-203 + buffer.py:95-105) in one launch.
        Returns (td float32[n], priority float32[n]) CUDA tensors."""
        torch = _torch()

        def f32(x):
            return torch.as_tensor(x).to(device=self.device, dtype=torch.float32).contiguous().reshape(-1)

        qo = torch.as_tensor(q_online).to(device=self.device, dtype=torch.float32).contiguous()
        qt = torch.as_tensor(q_target_next).to(device=self.device, dtype=torch.float32).contiguous()
        qn = None if q_online_next is None else torch.as_tensor(q_online_next).to(device=self.device, dtype=torch.float32).contiguous()
        a = torch.as_tensor(action).to(device=self.device, dtype=torch.int64).contiguous().reshape(-1)
        r, d, s = f32(reward), f32(done), f32(steps)
        ix = torch.as_tensor(idx).to(device=self.device, dtype=torch.int64).contiguous().reshape(-1)
        n = int(ix.numel())
        assert qo.shape == (n, 5) and qt.shape == (n, 5)
        td = torch.empty(n, dtype=torch.float32, device=self.device)
        pr = torch.empty(n, dtype=torch.float32, device=self.device)
        _native.check(self._lib.mapf_per_td_update(
            self._h, C.c_void_p(qo.data_ptr()), C.c_void_p(qt.data_ptr()), C.c_void_p(qn.data_ptr()) if qn is not None else None,
            C.c_void_p(a.data_ptr()), C.c_void_p(r.data_ptr()), C.c_void_p(d.data_ptr()), C.c_void_p(s.data_ptr()),
            C.c_void_p(ix.data_ptr()), n, float(gamma), float(alpha), int(old_ptr), int(ptr), int(slot_steps),
            C.c_void_p(td.data_ptr()), C.c_void_p(pr.data_ptr()), self._stream()))
        return td, pr   # asynchronous on the current stream

    def cycle(self, update=None, sample_size: int = 0, uniforms=None, beta=None, old_ptr=0, ptr=0,
              slot_steps=config.max_steps, gamma=0.99, alpha=config.prioritized_replay_alpha, out=None):
        """One learner cycle in ONE launch (mapf_per_cycle): `update` = dict(q_online f32[n,5], q_target_next f32[n,5],
        action i64[n], reward f32[n], done f32[n], steps f32[n], idx i64[n][, q_online_next]) of the batch that has just been
        through the two Q forwards -> its priorities go into the tree; then `sample_size` new transitions are drawn from
        the refreshed tree (uniforms f64[sample_size] in [0,1), default torch.rand) with IS weights when `beta` is given.
        All tensors are float32 / int64 CUDA tensors, used as they are (no conversion, no synchronisation); `out` may hold
        pre-allocated outputs (td, prio, idx, sample_prio, weights) for CUDA-graph capture.
        Returns dict(td, prio, idx, sample_prio, weights) (entries None for an empty half)."""
        torch = _torch()
        out = dict(out or {})
        a = _native.PerCycleArgs()
        n = 0
        if update is not None:
            ix = update["idx"]
            n = int(ix.numel())
            for k in ("q_online", "q_target_next", "reward", "done", "steps"):
                t = update[k]
                assert t.is_cuda and t.dtype == torch.float32 and t.is_contiguous(), k
            assert update["action"].dtype == torch.int64 and ix.dtype == torch.int64 and ix.is_contiguous()
            assert tuple(update["q_online"].shape) == (n, 5) and tuple(update["q_target_next"].shape) == (n, 5)
            out.setdefault("td", torch.empty(n, dtype=torch.float32, device=self.device))
            out.setdefault("prio", torch.empty(n, dtype=torch.float32, device=self.device))
            qn = update.get("q_online_next")
            a.d_q_online, a.d_q_target_next = update["q_online"].data_ptr(), update["q_target_next"].data_ptr()
            a.d_q_online_next = qn.data_ptr() if qn is not None else None
            a.d_action, a.d_reward, a.d_done = update["action"].data_ptr(), update["reward"].data_ptr(), update["done"].data_ptr()
            a.d_steps, a.d_idx = update["steps"].data_ptr(), ix.data_ptr()
            a.d_td_out, a.d_prio_out = out["td"].data_ptr(), out["prio"].data_ptr()
        a.n_update, a.gamma, a.alpha = n, float(gamma), float(alpha)
        a.old_ptr, a.ptr, a.slot_steps = int(old_ptr), int(ptr), int(slot_steps)
        m = int(sample_size)
        if m > 0:
            u = uniforms if uniforms is not None else torch.rand(m, dtype=torch.float64, device=self.device)
            assert u.is_cuda and u.dtype == torch.float64 and u.is_contiguous() and u.numel() == m
            out.setdefault("idx", torch.empty(m, dtype=torch.int64, device=self.device))
            out.setdefault("sample_prio", torch.empty(m, dtype=torch.float64, device=self.device))
            if beta is not None:
                out.setdefault("weights", torch.empty(m, dtype=torch.float32, device=self.device))
            a.d_uniforms, a.d_sample_idx_out, a.d_sample_prio_out = u.data_ptr(), out["idx"].data_ptr(), out["sample_prio"].data_ptr()
            a.d_sample_weight_out = out["weights"].data_ptr() if beta is not None else None
            out["_uniforms"] = u   # keep alive
        a.n_sample, a.beta = m, float(beta or 0.0)
        _native.check(self._lib.mapf_per_cycle(self._h, C.byref(a), self._stream()))
        for k in ("td", "prio", "idx", "sample_prio", "weights"):
            out.setdefault(k, None)
        return out

    def check(self):
        """Synchronous: IndexError if an update was handed a leaf index outside [0, capacity) since the last call (numpy
        raises at once; the kernels skip the entry and latch); AssertionError if a sample (`sample_device`, `cycle`)
        returned a leaf whose priority is not > 0 (the reference asserts at once, buffer.py:74; the kernels return the
        leaf the reference's descent finds, and the importance weights of that batch are undefined).  One condition is
        raised per call, the index one first; a second latched condition is raised by the next call."""
        _native.check(self._lib.mapf_per_status(self._h, self._stream()))

    # -- reference numpy API -------------------------------------------------------------------
    def batch_sample(self, batch_size: int):  # buffer.py:56-78
        # np.random.uniform(0, interval, B) == interval * np.random.random_sample(B): same global stream use
        u = np.random.random_sample(batch_size)
        idx, pr, _ = self.sample_device(batch_size, u)
        idxes, priorities = idx.cpu().numpy(), pr.cpu().numpy()
        assert np.all(priorities > 0), 'idx: {}, priority: {}'.format(idxes, priorities)
        assert np.all(idxes >= 0) and np.all(idxes < self.capacity)
        return idxes, priorities

    def batch_update(self, idxes: np.ndarray, priorities: np.ndarray):  # buffer.py:95-105
        leaf = np.array(idxes, dtype=np.int64, copy=True)
        if leaf.size and (leaf.min() < 0 or leaf.max() >= self.capacity):
            raise IndexError("leaf index outside [0, capacity)")   # what numpy's fancy assignment raises (buffer.py:97)
        idxes += self.capacity - 1  # the reference mutates the caller's array (buffer.py:96)
        self.update_device(leaf, np.asarray(priorities, dtype=np.float64))

    def update(self, idx: int, priority: float):  # buffer.py:80-93
        assert 0 <= idx < self.capacity
        self.update_device(np.asarray([idx], dtype=np.int64), np.asarray([priority], dtype=np.float64))


PrioritizedReplayTree = SumTree


def actor_td_errors(rew, q, act, size, capacity=config.max_steps, device=None, forward_steps=config.forward_steps,
                    gamma=0.99):
    """Batched LocalBuffer.finish TD (buffer.py:170-177) on the device: |sum_{j<forward_steps} gamma^j r[t+j] + max_a q - q[a_t]|
    (the reference hard-codes 0.99 and reads config.forward_steps, buffer.py:174-175).
    rew float[E,capacity] (already fp16-rounded), q float32[E,capacity,5], act uint8[E,capacity], size int32[E]
    -> float64[E,capacity] CUDA tensor."""
    torch = _torch()
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    r = torch.as_tensor(rew).to(device=dev, dtype=torch.float32).contiguous()
    qq = torch.as_tensor(q).to(device=dev, dtype=torch.float32).contiguous()
    a = torch.as_tensor(act).to(device=dev, dtype=torch.uint8).contiguous()
    s = torch.as_tensor(size).to(device=dev, dtype=torch.int32).contiguous()
    E = int(s.numel())
    assert r.shape == (E, capacity) and qq.shape == (E, capacity, 5) and a.shape == (E, capacity)
    td = torch.empty((E, capacity), dtype=torch.float64, device=dev)
    _native.check(_native.lib().mapf_actor_td_n(C.c_void_p(r.data_ptr()), C.c_void_p(qq.data_ptr()), C.c_void_p(a.data_ptr()),
                                                C.c_void_p(s.data_ptr()), E, capacity, int(forward_steps), float(gamma),
                                                C.c_void_p(td.data_ptr()),
                                                C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
    return td


class LocalBuffer:
    """buffer.LocalBuffer (buffer.py:108-179): per-episode storage with the reference's field names."""
    __slots__ = ('actor_id', 'map_len', 'num_agents', 'obs_buf', 'act_buf', 'rew_buf', 'hid_buf', 'comm_buf', 'q_buf',
                 'capacity', 'size', 'done', 'td_errors')

    def __init__(self, actor_id, num_agents, map_len, init_obs, size=config.max_steps):
        self.actor_id = actor_id
        self.num_agents = num_agents
        self.map_len = map_len
        self.obs_buf = np.zeros((size + 1, self.num_agents, *config.obs_shape), dtype=bool)
        self.act_buf = np.zeros((size), dtype=np.uint8)
        self.rew_buf = np.zeros((size), dtype=np.float16)
        self.hid_buf = np.zeros((size, self.num_agents, config.latent_dim), dtype=np.float16)
        self.comm_buf = np.zeros((size + 1, num_agents, num_agents), dtype=bool)
        self.q_buf = np.zeros((size + 1, 5), dtype=np.float32)
        self.capacity = size
        self.size = 0
        self.obs_buf[0] = init_obs

    def __len__(self):
        return self.size

    def add(self, q_val, action: int, reward, next_obs, hidden, comm_mask):  # buffer.py:140-151
        assert self.size < self.capacity
        self.act_buf[self.size] = action
        self.rew_buf[self.size] = reward
        self.obs_buf[self.size + 1] = next_obs
        self.q_buf[self.size] = q_val
        self.hid_buf[self.size] = hidden
        self.comm_buf[self.size] = comm_mask
        self.size += 1

    def finish(self, last_q_val=None, comm_mask=None):  # buffer.py:153-179
        if last_q_val is None:
            self.done = True
        else:
            self.done = False
            self.q_buf[self.size] = last_q_val
            self.comm_buf[self.size] = comm_mask
        cap = self.capacity
        rew = np.zeros((1, cap), dtype=np.float32)
        rew[0, :self.size] = self.rew_buf[:self.size].astype(np.float32)  # fp16 -> fp32 is exact
        q = np.zeros((1, cap, 5), dtype=np.float32)
        q[0, :self.size] = self.q_buf[:self.size]
        act = np.zeros((1, cap), dtype=np.uint8)
        act[0, :self.size] = self.act_buf[:self.size]
        td = actor_td_errors(rew, q, act, np.asarray([self.size], dtype=np.int32), capacity=cap)
        self.td_errors = td[0].cpu().numpy()

        self.obs_buf = self.obs_buf[:self.size + 1]
        self.act_buf = self.act_buf[:self.size]
        self.rew_buf = self.rew_buf[:self.size]
        self.hid_buf = self.hid_buf[:self.size]
        self.comm_buf = self.comm_buf[:self.size + 1]
        self.q_buf = self.q_buf[:self.size + 1]
        return (self.actor_id, self.num_agents, self.map_len, self.obs_buf, self.act_buf, self.rew_buf, self.hid_buf,
                self.td_errors, self.done, self.size, self.comm_buf)
