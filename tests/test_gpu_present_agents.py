"""GPU: present-agent batches.  mapf_obs_unpack_present equals the padded unpack indexed by the present rows (bit-exact, padding
rows zero); gather(idx, present=True) equals the padded gather indexed the same way on a compact and a dense store; the store's
per-slot agent count as add() and the actor write it; and padded / present-only twins of the actor and the learner agree."""
import copy
import ctypes as C

import numpy as np
import pytest

from mapf_rl_b200 import _native, packed
from mapf_rl_b200.present import PresentRows, present_np, unpack_obs_present

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _counts(kind, count, N, rng):
    if kind == "all1":
        return np.ones(count, dtype=np.int64)
    if kind == "allN":
        return np.full(count, N, dtype=np.int64)
    if kind == "alternating":
        return np.where(np.arange(count) % 2, N, 1).astype(np.int64)
    return rng.integers(1, N + 1, size=count).astype(np.int64)


def _unpack_present_raw(bits, rows, n8, first, out_rows, dtype, fill):
    """mapf_obs_unpack_present into an output pre-filled with `fill` (so rows the kernel leaves unwritten show)."""
    import torch
    code = {torch.uint8: _native.DTYPE_U8, torch.float16: _native.DTYPE_F16, torch.bfloat16: _native.DTYPE_BF16}[dtype]
    out = torch.full((out_rows, 6, 9, 9), fill, dtype=dtype, device=DEV)
    _native.check(_native.lib().mapf_obs_unpack_present(
        C.c_void_p(bits.data_ptr()), C.c_void_p(rows.data_ptr()), C.c_void_p(n8.data_ptr()), C.c_void_p(first.data_ptr()),
        int(rows.numel()), int(bits.shape[1]), out_rows, code, C.c_void_p(out.data_ptr()),
        C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return out


@pytest.mark.parametrize("N", [1, 6, 31, 32, 33, 64, 128])
def test_obs_unpack_present_equals_indexed_unpack(N):
    import torch
    rng = np.random.default_rng(N)
    g = torch.Generator(device=DEV)
    g.manual_seed(N)
    F = 8192 + 17
    bits = torch.randint(0, 256, (F, N, 64), dtype=torch.uint8, device=DEV, generator=g)   # pad bits set: ignored
    for count in (1, 2, 7, 8192 if N <= 33 else 1500):
        for kind in ("all1", "allN", "random", "alternating"):
            counts = _counts(kind, count, N, rng)
            first, index, M, M_pad = present_np(counts, N)
            rows = torch.as_tensor(rng.integers(0, F, size=count), dtype=torch.int64, device=DEV)
            pr = PresentRows(torch.as_tensor(counts, device=DEV), M, N)
            idx = torch.as_tensor(index, device=DEV)
            for dt in (torch.uint8, torch.float16, torch.bfloat16):
                want = packed.unpack_obs(bits, rows, dtype=dt).flatten(0, 1).index_select(0, idx)
                got = unpack_obs_present(bits, rows, pr, dtype=dt)
                assert got.dtype == dt and tuple(got.shape) == (M_pad, 6, 9, 9)
                assert torch.equal(got[:M].view(torch.uint8) if dt == torch.uint8 else got[:M].view(torch.int16),
                                   want.view(torch.uint8) if dt == torch.uint8 else want.view(torch.int16)), (N, count, kind, dt)
                # every row is written: padding rows and an odd output length (a short last run) included
                n8 = torch.as_tensor(counts.astype(np.uint8), device=DEV)
                f32 = torch.as_tensor(first, device=DEV)
                for out_rows in (M_pad, M + 3):
                    raw = _unpack_present_raw(bits, rows, n8, f32, out_rows, dt, 7)
                    assert torch.equal(raw[:M], got[:M]) and not raw[M:].any(), (N, count, kind, dt, out_rows)


def test_obs_unpack_present_clamps_counts_above_N():
    import torch
    N = 6
    bits = torch.randint(0, 256, (10, N, 64), dtype=torch.uint8, device=DEV)
    rows = torch.arange(3, dtype=torch.int64, device=DEV)
    n8 = torch.tensor([9, 2, 200], dtype=torch.uint8, device=DEV)      # 9 and 200 read as 6
    first = torch.tensor([0, 6, 8], dtype=torch.int32, device=DEV)
    out = _unpack_present_raw(bits, rows, n8, first, 24, torch.uint8, 7)
    want = packed.unpack_obs(bits, rows).flatten(0, 1)
    assert torch.equal(out[:6], want[:6]) and torch.equal(out[6:8], want[6:8]) and torch.equal(out[8:14], want[12:18])
    assert not out[14:].any()


def _agents_pair(N, latent, rng, counts):
    from test_gpu_compact_store import _store_pair
    cap, S = 8, 32
    sizes = [S, 1, 17, 3, S, 25, 16, 31]
    dones = [0, 1, 1, 0, 1, 0, 1, 0]
    d, c = _store_pair(N, latent, cap, S, rng, sizes, dones)
    import torch
    for s in (d, c):
        s.agents_buf.copy_(torch.as_tensor(np.asarray(counts, dtype=np.uint8)))
    idx = []
    for slot in range(cap):
        for t in sorted({0, 1, d.bt_steps - 1, d.bt_steps, sizes[slot] - 2, sizes[slot] - 1}):
            if 0 <= t < sizes[slot]:
                idx.append(slot * S + t)
    return d, c, idx, cap * S


@pytest.mark.parametrize("N,latent", [(6, 256), (1, 256), (13, 256), (33, 12), (8, 20)])
def test_gather_present_equals_indexed_gather(N, latent):
    import torch
    rng = np.random.default_rng(N * 7 + latent)
    counts = np.minimum(np.asarray([N, 1, 3, 2, N, 5, 1, 4]), N)
    d, c, idx_ok, leaves = _agents_pair(N, latent, rng, counts)
    idx_ok = np.asarray(idx_ok, dtype=np.int64)
    idx_bad = rng.integers(0, leaves, size=40)                     # includes leaves beyond their episode
    for sel, latch in ((idx_ok, 0), (np.concatenate([idx_ok, idx_bad]), 1)):
        idx = torch.as_tensor(sel, device=DEV)
        first, index, M, M_pad = present_np(counts[sel // d.max_steps], N)
        W = d.bt_steps + d.forward_steps
        for s in (d, c):
            s._err.zero_()
            ref = s.gather(idx)
            s._err.zero_()
            got = s.gather(idx, present=True)
            assert int(s._err.item()) == latch
            pr = got["present"]
            assert pr.M == M and pr.M_pad == M_pad and np.array_equal(pr.first.cpu().numpy(), first)
            ti = torch.as_tensor(index, device=DEV)
            want_obs = ref["obs"].transpose(1, 2).reshape(len(sel) * N, W, 6, 9, 9).index_select(0, ti)
            assert got["obs"].shape == (M_pad, W, 6, 9, 9) and got["hidden"].shape == (M_pad, latent)
            assert torch.equal(got["obs"][:M].view(torch.int16), want_obs.view(torch.int16)), (s.compact, N)
            assert torch.equal(got["hidden"][:M].view(torch.int16), ref["hidden"].index_select(0, ti).view(torch.int16))
            assert not got["obs"][M:].any() and not got["hidden"][M:].any()
            for k in ("comm_mask", "action", "reward", "done", "steps", "bt_steps"):
                assert torch.equal(got[k], ref[k]), k


def test_add_writes_agents_and_rejects_out_of_range():
    import torch
    from replay_cases import make_episode
    from mapf_rl_b200 import ReplayStore
    rng = np.random.default_rng(2)
    N, S = 6, 32
    for compact in (False, True):
        st = ReplayStore(4, max_num_agents=N, device=DEV, max_steps=S, compact=compact)
        assert (st.agents_buf.cpu().numpy() == N).all()
        eps = []
        for n, size in ((3, 5), (1, 9), (6, 4)):
            ep = list(make_episode(rng, 0, n, size, True, latent=256, cap=S))
            ep[6] = np.repeat(ep[6][:, :1], n, axis=1)
            eps.append(tuple(ep))
        st.add(eps)
        assert st.agents_buf.cpu().numpy().tolist() == [3, 1, 6, N]
        for bad_n in (0, N + 1):
            bad = list(eps[0])
            bad[1] = bad_n
            ptr = st.ptr
            with pytest.raises(ValueError):
                st.add([tuple(bad)])
            assert st.ptr == ptr
        assert st.nbytes == sum(t.numel() * t.element_size() for t in (
            (st.obs_bits, st.comm_bits) if compact else (st.obs_buf, st.comm_mask)) + (
            st.hid_buf, st.act_buf, st.rew_buf, st.done_buf, st.size_buf, st.agents_buf))


def _actor(sized, compact, present_only, net, B=64, N=6, L=40, S=16, seed=3, record=None):
    from mapf_rl_b200 import BatchedEnvironment, ReplayStore
    from mapf_rl_b200.actor import BatchedActor
    from mapf_rl_b200.curriculum import Curriculum
    env = BatchedEnvironment(B, N, L, device=DEV, sized=sized)
    cur = None
    if sized:
        cur = Curriculum(max_num_agents=N, max_map_length=L)
        for lv in [(1, 10), (2, 10), (1, 15), (3, 20), (6, 40), (4, 30), (5, 12)]:
            cur._add(lv)
    store = ReplayStore(2 * B, max_num_agents=N, device=DEV, max_steps=S, latent_dim=256, compact=compact)

    def on_episode(actor, ids, slots, size, done, td):
        if record is not None:
            n = actor.env.sizes[0].cpu().numpy() if sized else np.full(B, N)
            record.append((slots.copy(), n[ids].copy()))

    actor = BatchedActor(env, net, store, epsilon=0.2, seed=seed, density=0.2, max_steps=S, curriculum=cur,
                         present_only=present_only, on_episode=on_episode)
    return actor


class _Stub:
    def reset(self):
        pass

    def step(self, obs, comm, reset_mask=None, present=None):
        import torch
        B, N = comm.shape[:2]
        z = torch.zeros((B, N), dtype=torch.int64, device=comm.device)
        return z, torch.zeros((B, N, 5), device=comm.device), torch.zeros((B, N, 256), device=comm.device)


@pytest.mark.parametrize("sized", [False, True])
@pytest.mark.parametrize("present_only", [False, True])
def test_actor_writes_agents_buf(sized, present_only):
    rec = []
    actor = _actor(sized, True, present_only, _Stub(), record=rec)
    actor.run(3 * 16)
    assert actor.episodes >= 2 * actor.B
    agents = actor.store.agents_buf.cpu().numpy()
    # finished episodes: the last one published in each slot (the ring reuses slots) that no running episode holds now
    last = {}
    for slots, n in rec:
        last.update(zip(slots.tolist(), n.tolist()))
    running = set(actor._slot_host.tolist())
    done = sorted(s for s in last if s not in running)
    assert done
    assert np.array_equal(agents[done], [last[s] for s in done])
    if sized:
        assert any((n < actor.N).any() for _, n in rec)
    # running episodes: their slots carry the current counts
    cur = actor.env.sizes[0].cpu().numpy() if sized else np.full(actor.B, actor.N)
    assert np.array_equal(agents[actor._slot_host], cur)


@pytest.mark.parametrize("compact", [False, True])
def test_actor_twin_padded_and_present_only(compact):
    import torch
    from mapf_rl_b200.qnet import Network
    torch.manual_seed(0)
    base = Network().to(DEV).double()     # fp64: an argmax tie cannot flip an action between the two paths
    runs = []
    for present_only in (False, True):
        net = copy.deepcopy(base)
        actor = _actor(True, compact, present_only, net)
        actor.run(2 * 16 + 5)             # at least two episode boundaries per environment
        actor.env.check()
        actor.store.priority_tree.check()
        runs.append(actor)
    a, b = runs
    assert a.episodes == b.episodes >= 2 * a.B and a.resets == b.resets
    sa, sb = a.store, b.store
    bufs = ("obs_bits", "comm_bits") if compact else ("obs_buf", "comm_mask")
    for k in bufs + ("hid_buf", "act_buf", "rew_buf", "done_buf", "size_buf", "agents_buf"):
        x, y = getattr(sa, k), getattr(sb, k)
        assert torch.equal(x.view(torch.int16) if x.dtype == torch.float16 else x,
                           y.view(torch.int16) if y.dtype == torch.float16 else y), k
    assert sa.size == sb.size and sa.ptr == sb.ptr
    ta, tb = sa.priority_tree.tree, sb.priority_tree.tree
    assert torch.allclose(ta, tb, rtol=1e-6, atol=0)
    assert (sa.agents_buf < a.N).any()


def _clone_store(src):
    from mapf_rl_b200 import ReplayStore
    dst = ReplayStore(src.capacity, max_num_agents=src.max_num_agents, device=DEV, max_steps=src.max_steps,
                      latent_dim=src.latent_dim, compact=src.compact)
    for k, v in vars(src).items():
        if hasattr(v, "copy_") and hasattr(dst, k):
            getattr(dst, k).copy_(v)
    dst.priority_tree.tree.copy_(src.priority_tree.tree)
    dst.size, dst.ptr, dst.counter, dst._size_host = src.size, src.ptr, src.counter, src._size_host.copy()
    return dst


@pytest.mark.parametrize("compact", [False, True])
def test_learner_twin_padded_and_present_only(compact):
    import torch
    from mapf_rl_b200.learner import BatchedLearner
    from mapf_rl_b200.qnet import Network
    torch.manual_seed(1)
    actor = _actor(True, compact, False, Network().to(DEV))
    actor.run(3 * 16)
    sa = actor.store
    sb = _clone_store(sa)
    assert len(sa) >= 256
    base = Network().to(DEV).double()
    init = {k: v.clone() for k, v in base.state_dict().items()}
    la = BatchedLearner(copy.deepcopy(base), sa, batch_size=64, seed=9, autocast_dtype=torch.float64)
    lb = BatchedLearner(copy.deepcopy(base), sb, batch_size=64, seed=9, autocast_dtype=torch.float64, present_only=True)
    for _ in range(3):
        xa, xb = la.update(want_stats=True), lb.update(want_stats=True)
        assert abs(xa["loss"] - xb["loss"]) <= 1e-5 * abs(xa["loss"])
        assert abs(xa["td_abs_mean"] - xb["td_abs_mean"]) <= 1e-5 * abs(xa["td_abs_mean"])
        # every sampled TD through its priority
        assert torch.allclose(sa.priority_tree.tree, sb.priority_tree.tree, rtol=1e-5, atol=0)
        assert torch.equal(la._next[0], lb._next[0])          # the same next batch
    pa, pb = la.model.state_dict(), lb.model.state_dict()
    for k in pa:
        moved = (pa[k] - init[k]).norm()
        assert (pb[k] - pa[k]).norm() <= 1e-3 * moved + 1e-12, k
