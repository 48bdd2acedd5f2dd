"""BatchedLearner — the reference learner's update (Learner.train, worker.py:282-340) with everything but the Q-network's
GEMMs / convolutions in this package's kernels, and nothing leaving the device:

    batch  = window gather of the transitions drawn in the PREVIOUS cycle            worker.py:106-184  (replay_gather kernel)
    q_tgt  = tar_model.bootstrap(obs[18 frames], bt + steps)                         worker.py:300-302  (PyTorch)
    q      = model.bootstrap(obs[16 frames], bt)                                     worker.py:304      (PyTorch)
    loss   = mean(w * huber(q[a] - (r + 0.99^steps (1 - done) max q_tgt)))           worker.py:306-310  (PyTorch, autograd)
    Adam step, grad clip 40, MultiStepLR, target sync every 2500 updates             worker.py:316-338  (PyTorch)
    ONE launch (mapf_per_cycle): TD -> priority -> stale mask -> leaf = p^alpha -> ancestors of THIS batch, then the NEXT
    batch's stratified sample + importance weights from the refreshed tree           worker.py:186-203, 114, 165-166

The reference ships (idx, priorities) to the buffer process and the next batch back through Ray; here the indices never leave
the device and the cycle has no host synchronisation (the only `.item()` calls are the optional statistics).  Mixed
precision: the reference runs fp16 autocast with a GradScaler (worker.py:283,316-323); on a B200 the same region runs under
bf16 autocast, which needs no loss scaling.  With more than one rank the gradients are averaged with ONE NCCL all-reduce of
the flattened 2.05 M fp32 gradients (8.2 MB) per update -- the only collective of the whole package.

`present_only=True` gathers each batch in present-agent rows (`ReplayStore.gather(idx, present=True)`) and runs both
bootstraps with the encoder on those rows only.  Sizing that batch reads its row count on the host when it is gathered, so the
host waits for update k's sampling before it can enqueue update k + 1 (DESIGN.md §4 measures what that costs).
"""
from __future__ import annotations

import copy
from typing import Optional

from . import config
from .replay import ReplayStore


def _torch():
    import torch
    return torch


class BatchedLearner:
    def __init__(self, model, store: ReplayStore, batch_size: int = config.batch_size, lr: float = 1e-4, gamma: float = 0.99,
                 grad_clip: float = 40.0, target_update_freq: int = 2500, autocast_dtype=None, allreduce: bool = False,
                 seed: int = 0, present_only: bool = False):
        torch = _torch()
        self.model, self.store, self.batch_size = model, store, int(batch_size)
        self.dev = store.device
        self.tar_model = copy.deepcopy(model).eval()                       # worker.py:258
        for p in self.tar_model.parameters():
            p.requires_grad_(False)
        self.optimizer = torch.optim.Adam(self.model.parameters(), lr=lr)   # worker.py:260
        self.scheduler = torch.optim.lr_scheduler.MultiStepLR(self.optimizer, milestones=[100000, 300000], gamma=0.5)  # :261
        self.gamma, self.grad_clip, self.target_update_freq = float(gamma), float(grad_clip), int(target_update_freq)
        self.autocast_dtype = autocast_dtype if autocast_dtype is not None else torch.bfloat16
        self.allreduce = bool(allreduce)
        self.gen = torch.Generator(device=self.dev)
        self.gen.manual_seed(seed)
        self.counter = 0
        self.loss = None
        self.present_only = bool(present_only)
        # (idx int64[B], weights f32[B], old_ptr, gathered batch) drawn by the previous cycle.  The window gather runs right
        # after the draw -- the reference's sample_batch assembles the batch under the buffer lock at sampling time,
        # worker.py:112-184 -- so an episode slot the actor evicts between two updates cannot tear the batch; its priorities
        # are then discarded by the stale-slot window [old_ptr, ptr) like the reference's (worker.py:192-201)
        self._next = None

    # -- the first batch of a run: the sample half of the cycle kernel alone ---------------------------------------------------
    def _first_sample(self):
        torch = _torch()
        u = torch.rand(self.batch_size, dtype=torch.float64, device=self.dev, generator=self.gen)
        out = self.store.priority_tree.cycle(sample_size=self.batch_size, uniforms=u, beta=self.store.beta)
        self._next = (out["idx"], out["weights"], self.store.ptr, self.store.gather(out["idx"], present=self.present_only))

    @staticmethod
    def huber(td, kappa: float = 1.0):   # worker.py:341-344
        a = td.abs()
        return _torch().where(a < kappa, 0.5 * a * a, a - 0.5)

    def _allreduce_grads(self):
        torch = _torch()
        import torch.distributed as dist
        if not (self.allreduce and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1):
            return
        grads = [p.grad for p in self.model.parameters() if p.grad is not None]
        flat = torch._utils._flatten_dense_tensors(grads)
        dist.all_reduce(flat, op=dist.ReduceOp.SUM)
        flat.div_(dist.get_world_size())
        for g, f in zip(grads, torch._utils._unflatten_dense_tensors(flat, grads)):
            g.copy_(f)

    def update(self, want_stats: bool = False):
        """One learner update (worker.py:287-338).  Asynchronous on the current stream unless `want_stats`."""
        torch = _torch()
        st, B = self.store, self.batch_size
        fwd = st.forward_steps
        if self._next is None:
            self._first_sample()
        idx, weights, old_ptr, b = self._next                               # batch assembled at sampling time (worker.py:118-162)
        obs, comm, hidden, pr = b["obs"], b["comm_mask"], b["hidden"], b.get("present")
        action = b["action"].unsqueeze(1)
        reward, done, steps = b["reward"].float().unsqueeze(1), b["done"].float().unsqueeze(1), b["steps"].float().unsqueeze(1)
        bt = b["bt_steps"]
        next_bt = bt + b["steps"].long()                                    # worker.py:296-297
        with torch.autocast("cuda", dtype=self.autocast_dtype):
            with torch.no_grad():
                q_tgt_all = self.tar_model.bootstrap(obs, next_bt, hidden, comm, present=pr).float()          # :302
            q_all = self.model.bootstrap(obs[:, :-fwd], bt, hidden, comm[:, :-fwd], present=pr).float()      # :304
        q_ = (1.0 - done) * q_tgt_all.max(1, keepdim=True)[0]
        td = q_all.gather(1, action) - (reward + torch.pow(self.gamma, steps) * q_)                           # :306
        loss = (weights.unsqueeze(1) * self.huber(td)).mean()                                                # :310
        self.optimizer.zero_grad(set_to_none=False)
        loss.backward()
        self._allreduce_grads()
        torch.nn.utils.clip_grad_norm_(self.model.parameters(), self.grad_clip)                              # :319
        self.optimizer.step()
        self.scheduler.step()
        # priorities of this batch in, next batch out: ONE launch, no host round trip (worker.py:308,331 + 114,165-166)
        u = torch.rand(B, dtype=torch.float64, device=self.dev, generator=self.gen)
        out = st.priority_tree.cycle(
            update=dict(q_online=q_all.detach().contiguous(), q_target_next=q_tgt_all.contiguous(), action=b["action"].contiguous(),
                        reward=reward.reshape(-1).contiguous(), done=done.reshape(-1).contiguous(),
                        steps=steps.reshape(-1).contiguous(), idx=idx),
            sample_size=B, uniforms=u, beta=st.beta, old_ptr=old_ptr, ptr=st.ptr, slot_steps=st.max_steps, gamma=self.gamma,
            alpha=st.alpha)
        self._next = (out["idx"], out["weights"], st.ptr, st.gather(out["idx"], present=self.present_only))
        self.counter += 1
        if self.counter % self.target_update_freq == 0:                                                      # :336-337
            self.tar_model.load_state_dict(self.model.state_dict())
        if want_stats:
            # synchronising anyway: surface a latched tree condition (a sampled leaf of priority 0 would make the next
            # batch's importance weights NaN or 0, and the loss takes them as they are)
            st.priority_tree.check()
            self.loss = float(loss.item())
            return dict(loss=self.loss, td_abs_mean=float(out["td"].abs().mean().item()),
                        prio_min=float(out["prio"].min().item()), kernel_td_vs_torch=float((out["td"] - td.detach().reshape(-1)).abs().max().item()))
        return None

    def ready(self, min_transitions: Optional[int] = None) -> bool:
        """worker.py:228-232: enough stored transitions to start learning (config.learning_starts by default)."""
        need = config.learning_starts if min_transitions is None else int(min_transitions)
        return len(self.store) >= max(need, self.batch_size)
