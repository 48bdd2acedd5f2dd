"""GPU: the replay store's window gathers against the host restatement tests/replay_window_ref.py, bit for bit.

mapf_replay_gather (dense store), mapf_replay_gather_compact and mapf_replay_gather_present (compact store) are called through
the C ABI at every window geometry of replay_window_ref.GEOMETRIES, on stores whose ring has wrapped (shorter episodes over
full ones), at every edge step of every slot, at random and repeated leaves, with leaves past their episode (the error
word), with present-row outputs of any length, at the largest batch the ABI serves and past it, and with sampled rows and
outputs past 2^32 bytes.  Every output is pre-filled with 0xFF bytes (fp16 NaN) and followed by a guard of sentinel bytes,
so an element a kernel skips and a write past the output both fail.

The test_offset64_* cases need up to about 10 GB of device memory; `-k "not offset64"` deselects them on a small GPU."""
import ctypes as C

import numpy as np
import pytest

import replay_window_ref as wr
from mapf_rl_b200 import _native, packed
from mapf_rl_b200.present import present_np
from replay_cases import ring_episodes

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
FILL, GUARD_BYTE, GUARD = 0xFF, 0xA5, 4096
FIELDS = ("obs", "comm_mask", "hidden", "action", "reward", "done", "steps", "bt_steps")


@pytest.fixture
def pow2_tree(monkeypatch):
    """ReplayStore with any slot count and max_steps: its sum tree (the reference's takes a power-of-two capacity only) gets
    the next power of two.  The gathers never read the tree; leaves past the store's keep priority 0."""
    from mapf_rl_b200 import replay
    from mapf_rl_b200.buffer import SumTree

    class Pow2Tree(SumTree):
        def __init__(self, capacity, device=None):
            super().__init__(1 << (int(capacity) - 1).bit_length(), device=device)

    monkeypatch.setattr(replay, "SumTree", Pow2Tree)


def _store(geo, cap, compact):
    from mapf_rl_b200 import ReplayStore
    return ReplayStore(cap, max_num_agents=geo.N, device=DEV, max_steps=geo.S, bt_steps=geo.bt, forward_steps=geo.fwd,
                       latent_dim=geo.latent, compact=compact)


class Out:
    """The outputs of one gather call, each filled with FILL and followed by GUARD bytes of GUARD_BYTE."""

    def __init__(self, geo, B, out_rows=None):
        import torch
        N, W = geo.N, geo.bt + geo.fwd
        rows = B * N if out_rows is None else out_rows
        obs = (B, W, N, 6, 9, 9) if out_rows is None else (out_rows, W, 6, 9, 9)
        shapes = dict(obs=(obs, torch.float16), comm_mask=((B, W, N, N), torch.uint8), hidden=((rows, geo.latent), torch.float16),
                      action=((B,), torch.int64), reward=((B,), torch.float16), done=((B,), torch.float16),
                      steps=((B,), torch.float16), bt_steps=((B,), torch.int64))
        self.raw, self.t = {}, {}
        for k, (shape, dt) in shapes.items():
            n = int(np.prod(shape)) * torch.empty(0, dtype=dt).element_size()
            buf = torch.full((n + GUARD,), FILL, dtype=torch.uint8, device=DEV)
            buf[n:] = GUARD_BYTE
            self.raw[k] = (buf, n)
            self.t[k] = buf[:n].view(dt).view(shape)
        self.batch = _native.ReplayBatch(*[self.t[k].data_ptr() for k in FIELDS])

    def guards_intact(self):
        return all(bool((buf[n:] == GUARD_BYTE).all()) for buf, n in self.raw.values())

    def untouched(self):
        return all(bool((buf[:n] == FILL).all()) for buf, n in self.raw.values())

    def host(self, k, sl=slice(None)):
        x = self.t[k][sl].cpu().numpy()
        return x.view(np.uint16) if x.dtype == np.float16 else x


def _gather(kind, store, idx, first=None, out_rows=None):
    """One call of mapf_replay_gather ("dense"), _compact or _present into fresh `Out` tensors -> (code, Out, error word)."""
    import torch
    geo = wr.Geometry(store.max_num_agents, store.max_steps, store.bt_steps, store.forward_steps, store.latent_dim)
    B = int(idx.numel())
    out = Out(geo, B, out_rows if kind == "present" else None)
    err = torch.zeros(1, dtype=torch.int32, device=DEV)
    lib, view, p = _native.lib(), store._view(), lambda t: C.c_void_p(t.data_ptr())
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    if kind == "dense":
        code = lib.mapf_replay_gather(C.byref(view), p(idx), B, C.byref(out.batch), p(err), s)
    elif kind == "compact":
        code = lib.mapf_replay_gather_compact(C.byref(view), p(idx), B, C.byref(out.batch), p(err), s)
    else:
        code = lib.mapf_replay_gather_present(C.byref(view), p(store.agents_buf), p(idx), p(first), B, out_rows,
                                              C.byref(out.batch), p(err), s)
    torch.cuda.synchronize()
    return code, out, int(err.item())


def _u16(x):
    x = np.ascontiguousarray(x)
    return x.view(np.uint16) if x.dtype == np.float16 else x


def _assert_scalars(host, ref):
    for k in ("action", "reward", "done", "steps", "bt_steps"):
        assert np.array_equal(host(k), _u16(ref[k])), k


def _assert_out(out, ref, present=None):
    """`out` equals gather_ref's batch `ref` (present: present_ref's (obs, hidden) for the obs / hidden rows), guards intact."""
    obs, hidden = (ref["obs"], ref["hidden"]) if present is None else present
    assert np.array_equal(out.host("obs"), _u16(obs))
    assert np.array_equal(out.host("hidden"), _u16(hidden))
    assert np.array_equal(out.host("comm_mask"), ref["comm_mask"])
    _assert_scalars(out.host, ref)
    assert out.guards_intact()


def _assert_dict(got, ref, present=None):
    obs, hidden = (ref["obs"], ref["hidden"]) if present is None else present
    h = lambda k: _u16(got[k].cpu().numpy())
    assert np.array_equal(h("obs"), _u16(obs)) and np.array_equal(h("hidden"), _u16(hidden))
    assert np.array_equal(h("comm_mask"), ref["comm_mask"])
    _assert_scalars(h, ref)


def _mirror(geo, cap, eps, compact, agents_over):
    """Host slots of what ReplayStore.add leaves in a fresh store: a dense store writes agents < n of each frame and row,
    a compact one zeros the rest and keeps one hidden vector per transition.  agents_over: {slot: agents entry} set after."""
    N, S = geo.N, geo.S
    obs = np.zeros(((S + 1) * cap, N, 6, 9, 9), dtype=np.uint8)
    comm = np.zeros(((S + 1) * cap, N, N), dtype=np.uint8)
    hid = np.zeros((S * cap, N, geo.latent), dtype=np.float16)
    act, rew = np.zeros(S * cap, dtype=np.uint8), np.zeros(S * cap, dtype=np.float16)
    done, size, agents = np.zeros(cap, dtype=bool), np.zeros(cap, dtype=np.int64), np.full(cap, N)
    for k, ep in enumerate(eps):
        g, n, T = k % cap, ep[1], ep[9]
        f, r = g * (S + 1), g * S
        if compact:
            obs[f:f + T + 1], comm[f:f + T + 1] = 0, 0
            hid[r:r + T] = ep[6][:, :1]
        else:
            hid[r:r + T, :n] = ep[6]
        obs[f:f + T + 1, :n] = ep[3]
        comm[f:f + T + 1, :n, :n] = ep[10]
        act[r:r + T], rew[r:r + T] = ep[4], ep[5]
        done[g], size[g], agents[g] = ep[8], T, n
    for g, v in agents_over.items():
        agents[g] = v
    return {g: wr.slot_of(obs, comm, hid, act, rew, done, size, agents, g, S) for g in range(cap)}


def _ring_pair(geo, seed):
    """A dense and a compact store filled with the same ring_episodes, the last slot's agents entry set above N ->
    (dense, compact, {"dense": slots, "compact": slots}, rng)."""
    rng = np.random.default_rng(seed)
    cap, eps = ring_episodes(geo, rng)
    d, c = _store(geo, cap, False), _store(geo, cap, True)
    d.add(eps)
    c.add(eps)
    for s in (d, c):
        s.agents_buf[cap - 1] = 255
    slots = {"dense": _mirror(geo, cap, eps, False, {cap - 1: 255}), "compact": _mirror(geo, cap, eps, True, {cap - 1: 255})}
    assert d.size_buf.cpu().tolist() == [slots["dense"][g].size for g in range(cap)]
    return d, c, slots, rng


def _leaves(slots, geo, rng, extra=24):
    """Every edge step of every slot, `extra` random leaves inside their episodes and some repeats, shuffled."""
    S = geo.S
    edges = [g * S + t for g in slots for t in wr.edge_steps(slots[g].size, geo)]
    valid = np.asarray([g * S + t for g in slots for t in range(slots[g].size)], dtype=np.int64)
    idx = np.concatenate([edges, rng.choice(valid, size=extra), edges[::3]]).astype(np.int64)
    rng.shuffle(idx)
    return idx


def _dev(x):
    import torch
    return torch.as_tensor(np.array(x)).to(DEV)


@pytest.mark.parametrize("geo", wr.GEOMETRIES, ids=lambda g: "x".join(map(str, g)))
def test_gathers_equal_reference(geo, pow2_tree):
    import torch
    d, c, slots, rng = _ring_pair(geo, 17 * sum(geo))
    W, S = geo.bt + geo.fwd, geo.S
    idx = _leaves(slots["dense"], geo, rng)
    ti = _dev(idx)
    ref = {k: wr.gather_ref(slots[k], idx, geo) for k in slots}
    for kind, store in (("dense", d), ("compact", c)):
        code, out, err = _gather(kind, store, ti)
        assert code == 0 and err == 0, kind
        _assert_out(out, ref[kind])
    _, _, first, M, M_pad = wr.present_ref(ref["compact"], geo)
    tf = _dev(first)
    if W <= wr.PRESENT_MAX_W:
        # any output length: exact, a short last run of rows, padding rows, and fewer rows than the batch has
        for rows in sorted({M_pad, M, M + 1, M + 7, M - 3} - {0}):
            code, out, err = _gather("present", c, ti, tf, rows)
            assert code == 0 and err == 0, rows
            _assert_out(out, ref["compact"], wr.present_ref(ref["compact"], geo, rows)[:2])
    else:
        code, out, err = _gather("present", c, ti, tf, M_pad)
        assert code == _native.MAPF_EINVAL and err == 0 and out.untouched()
        with pytest.raises(_native.MapfError) as e:
            c.gather(ti, present=True)
        assert e.value.code == _native.MAPF_EINVAL
    # the same through ReplayStore.gather; present rows of a compact store come from the kernel, a dense store's from its
    # padded gather indexed by PresentRows, both with the agents entry above N read as N
    for kind, store in (("compact", c), ("dense", d)):
        _assert_dict(store.gather(ti), ref[kind])
        if W <= wr.PRESENT_MAX_W:
            got = store.gather(ti, present=True)
            assert np.array_equal(got["present"].first.cpu().numpy(), first) and got["present"].M == M
            _assert_dict(got, ref[kind], wr.present_ref(ref[kind], geo)[:2])
        assert int(store._err.item()) == 0

    # leaves past their episode (stale frames and rows of a longer episode, or never written) latch the error word
    bad = np.asarray([g * S + t for g, sl in slots["dense"].items() if sl.size < S for t in {sl.size, S - 1}], dtype=np.int64)
    if not len(bad):
        return                           # every slot holds a full episode (max_steps 1)
    mixed = np.concatenate([idx[:20], bad])
    rng.shuffle(mixed)
    tm = _dev(mixed)
    ref = {k: wr.gather_ref(slots[k], mixed, geo) for k in slots}
    assert ref["dense"]["bad"].any()
    kinds = [("dense", d, None), ("compact", c, None)]
    if W <= wr.PRESENT_MAX_W:
        kinds.append(("present", c, wr.present_ref(ref["compact"], geo)))
    for kind, store, pres in kinds:
        first_m = None if pres is None else _dev(pres[2])
        code, out, err = _gather(kind, store, tm, first_m, None if pres is None else pres[4])
        assert code == 0 and err == 1, kind
        _assert_out(out, ref["compact" if kind == "present" else kind], None if pres is None else pres[:2])
    # sample_batch(check=True) raises on such a leaf and clears the word; leaves inside their episodes pass
    leaves = np.arange(len(slots["dense"]) * S, dtype=np.int64)
    u = rng.uniform(0.05, 0.95, size=len(bad))
    for kind, store in (("dense", d), ("compact", c)):
        store.priority_tree.batch_update(leaves.copy(), np.zeros(len(leaves)))
        store.priority_tree.batch_update(bad.copy(), np.ones(len(bad)))
        with pytest.raises(AssertionError):
            store.sample_batch(len(bad), u)
        assert int(store._err.item()) == 0
        edges = np.unique(idx)
        store.priority_tree.batch_update(bad.copy(), np.zeros(len(bad)))
        store.priority_tree.batch_update(edges.copy(), np.ones(len(edges)))
        got = store.sample_batch(len(edges), rng.uniform(0.05, 0.95, size=len(edges)))
        assert np.array_equal(got[8], edges) and int(store._err.item()) == 0
        want = wr.gather_ref(slots[kind], edges, geo)
        assert np.array_equal(_u16(got[0].cpu().numpy()), _u16(want["obs"]))
        assert torch.equal(got[7].cpu(), torch.as_tensor(want["comm_mask"]).bool())


@pytest.mark.parametrize("N", [1, 3, 8, 127, 128])
def test_obs_unpack_present_any_out_rows(N):
    """mapf_obs_unpack_present at output lengths that are not a multiple of its 32-row runs, in every element type: rows of
    present agents, zeros up to out_rows, nothing past it."""
    import torch
    rng = np.random.default_rng(N)
    F, count = 40, 37
    raw = rng.integers(0, 256, size=(F, N, 64), dtype=np.uint8)          # pad bits set: ignored
    rows = rng.integers(0, F, size=count).astype(np.int64)
    n = rng.integers(1, N + 1, size=count)
    n[::6] = 255                                                          # above N: N rows
    first, index, M, _ = present_np(np.minimum(n, N), N)
    want = packed.unpack_obs_np(raw[rows]).reshape(count * N, 6, 9, 9)[index]
    lib, p = _native.lib(), lambda t: C.c_void_p(t.data_ptr())
    bits, trows, tn, tf = _dev(raw), _dev(rows), _dev(n.astype(np.uint8)), _dev(first)
    for dt, code, one in ((torch.uint8, _native.DTYPE_U8, 1), (torch.float16, _native.DTYPE_F16, 0x3C00),
                          (torch.bfloat16, _native.DTYPE_BF16, 0x3F80)):
        for out_rows in sorted(r for r in {M - 3, M + 1, M + 5, M + 13, M + 33} if r % 32):
            esz = torch.empty(0, dtype=dt).element_size()
            nb = out_rows * 486 * esz
            buf = torch.full((nb + GUARD,), FILL, dtype=torch.uint8, device=DEV)
            buf[nb:] = GUARD_BYTE
            rc = lib.mapf_obs_unpack_present(p(bits), p(trows), p(tn), p(tf), count, N, out_rows, code, p(buf),
                                             C.c_void_p(torch.cuda.current_stream().cuda_stream))
            assert rc == 0
            exp = np.zeros((out_rows, 6, 9, 9), dtype=np.uint8 if esz == 1 else np.uint16)
            exp[:min(M, out_rows)] = want[:out_rows].astype(exp.dtype) * one
            got = buf[:nb].cpu().numpy().view(exp.dtype).reshape(exp.shape)
            assert np.array_equal(got, exp), (dt, out_rows)
            assert bool((buf[nb:] == GUARD_BYTE).all()), (dt, out_rows)


def test_batch_limit(pow2_tree):
    """65,535 samples (gridDim.y of the dense and compact kernels) against the reference; 65,536 refused by all three
    entry points with nothing written."""
    geo = wr.Geometry(1, 4, 1, 1, 8)
    d, c, slots, rng = _ring_pair(geo, 3)
    valid = np.asarray([g * geo.S + t for g, sl in slots["dense"].items() for t in range(sl.size)], dtype=np.int64)
    B = 65535
    idx = rng.choice(valid, size=B)
    ti = _dev(idx)
    ref = {k: wr.gather_ref(slots[k], idx, geo) for k in slots}
    for kind, store in (("dense", d), ("compact", c)):
        code, out, err = _gather(kind, store, ti)
        assert code == 0 and err == 0
        _assert_out(out, ref[kind])
    pres = wr.present_ref(ref["compact"], geo)
    code, out, err = _gather("present", c, ti, _dev(pres[2]), pres[4])
    assert code == 0 and err == 0
    _assert_out(out, ref["compact"], pres[:2])
    del out
    t2 = _dev(np.concatenate([idx, idx[:1]]))
    first2 = _dev(np.arange(B + 1, dtype=np.int32))
    for kind, store in (("dense", d), ("compact", c), ("present", c)):
        code, out, err = _gather(kind, store, t2, first2, B + 1)
        assert code == _native.MAPF_EINVAL and err == 0 and out.untouched(), kind


def _random_slot(rng, geo, size, done, agents):
    """One slot with every frame and row random, also past `size` (what the gathers must not serve as live), and random
    observation and comm-mask pad bits -> (Slot, obs_bits, comm_bits)."""
    N, S = geo.N, geo.S
    obs_bits = rng.integers(0, 256, size=(S + 1, N, 64), dtype=np.uint8)
    comm_bits = rng.integers(0, 256, size=(S + 1, N, packed.comm_bytes(N)), dtype=np.uint8)
    hid = rng.standard_normal((S, geo.latent)).astype(np.float16)
    slot = wr.Slot(packed.unpack_obs_np(obs_bits), packed.unpack_comm(comm_bits, N),
                   np.broadcast_to(hid[:, None], (S, N, geo.latent)), rng.integers(0, 5, size=S).astype(np.uint8),
                   rng.standard_normal(S).astype(np.float16), done, size, agents)
    return slot, obs_bits, comm_bits


def _write_slot(store, g, slot, obs_bits, comm_bits):
    """Slot g's device rows, written in place (a store of many GB is never copied to the host)."""
    S = store.max_steps
    f, r = slice(g * (S + 1), (g + 1) * (S + 1)), slice(g * S, (g + 1) * S)
    if store.compact:
        store.obs_bits[f] = _dev(obs_bits)
        store.comm_bits[f] = _dev(comm_bits)
        store.hid_buf[r] = _dev(slot.hidden[:, 0])
    else:
        store.obs_buf[f] = _dev(slot.obs)
        store.comm_mask[f] = _dev(slot.comm)
        store.hid_buf[r] = _dev(slot.hidden)
    store.act_buf[r] = _dev(slot.action)
    store.rew_buf[r] = _dev(slot.reward)
    store.done_buf[g] = int(slot.done)
    store.size_buf[g] = slot.size
    store.agents_buf[g] = slot.agents


def _fill_last_slots(store, geo, rng, k):
    """Random episodes in the last k slots (sizes S, S - 1, 1, bt, ...) -> their host slots."""
    cap, S = store.capacity, geo.S
    sizes = [S, S - 1, 1, geo.bt, geo.bt + 1, 2] + [int(x) for x in rng.integers(1, S + 1, size=k)]
    slots = {}
    for j, g in enumerate(range(cap - k, cap)):
        slot, ob, cb = _random_slot(rng, geo, sizes[j], j % 2 == 0, int(rng.integers(1, geo.N + 1)))
        _write_slot(store, g, slot, ob, cb)
        slots[g] = slot
    return slots


@pytest.mark.parametrize("compact", [False, True])
def test_offset64_store_rows(compact, pow2_tree):
    """Sampled rows past 2^32 bytes into the store: a dense store of 1,100 slots at N = 32 (obs_buf 4.4 GB, hid_buf 4.6 GB)
    and a compact one of 2,100 slots at N = 128 (obs_bits 4.4 GB), the last 8 slots sampled."""
    geo = wr.Geometry(128 if compact else 32, 256, 16, 2, 256)
    cap = 2100 if compact else 1100
    store = _store(geo, cap, compact)
    rng = np.random.default_rng(cap)
    slots = _fill_last_slots(store, geo, rng, 8)
    g0, S, N = min(slots), geo.S, geo.N
    if compact:
        assert g0 * (S + 1) * N * 64 > 2 ** 32
    else:
        assert g0 * (S + 1) * N * 486 > 2 ** 32 and g0 * S * N * geo.latent * 2 > 2 ** 32
    idx = _leaves(slots, geo, rng, extra=16)
    ti = _dev(idx)
    ref = wr.gather_ref(slots, idx, geo)
    code, out, err = _gather("compact" if compact else "dense", store, ti)
    assert code == 0 and err == 0
    _assert_out(out, ref)
    del out
    pres = wr.present_ref(ref, geo)
    if compact:
        code, out, err = _gather("present", store, ti, _dev(pres[2]), pres[4])
        assert code == 0 and err == 0
        _assert_out(out, ref, pres[:2])
        del out
    _assert_dict(store.gather(ti, present=True), ref, pres[:2])


def test_offset64_output(pow2_tree):
    """Outputs past 2^32 bytes: N = 128, W = 18, B = 2,048 (4.6 GB of fp16 observations) from each of the three gathers;
    the samples (present rows) that reach past 2^32 compared in full, every sample's scalars."""
    import torch
    geo = wr.Geometry(128, 256, 16, 2, 256)
    N, W, B = geo.N, geo.bt + geo.fwd, 2048
    rng = np.random.default_rng(2048)
    d, c = _store(geo, 4, False), _store(geo, 4, True)
    slots = {}
    for g in range(4):
        slot, ob, cb = _random_slot(rng, geo, geo.S - g, g % 2 == 1, 255 if g == 0 else N)
        _write_slot(d, g, slot, ob, cb)
        _write_slot(c, g, slot, ob, cb)
        slots[g] = slot
    valid = np.asarray([g * geo.S + t for g, sl in slots.items() for t in range(sl.size)], dtype=np.int64)
    idx = rng.choice(valid, size=B)
    ti = _dev(idx)
    sc = wr.scalars_ref(slots, idx, geo)
    sample = W * N * 486 * 2
    b0 = 2 ** 32 // sample                    # first sample whose observations reach past 2^32 bytes
    assert B * sample > 2 ** 32 and b0 < B
    tail = wr.gather_ref(slots, idx[b0:], geo)
    for kind, store in (("dense", d), ("compact", c)):
        code, out, err = _gather(kind, store, ti)
        assert code == 0 and err == 0, kind
        _assert_scalars(out.host, sc)
        assert np.array_equal(out.host("obs", slice(b0, None)), _u16(tail["obs"])), kind
        assert np.array_equal(out.host("comm_mask", slice(b0, None)), tail["comm_mask"]), kind
        assert np.array_equal(out.host("hidden", slice(b0 * N, None)), _u16(tail["hidden"])), kind
        assert out.guards_intact(), kind
        del out
        torch.cuda.empty_cache()
    # present rows: all N agents of every sample, so M = B * N rows
    first = np.arange(B, dtype=np.int32) * N
    row = W * 486 * 2
    r0 = 2 ** 32 // row
    assert B * N * row > 2 ** 32
    code, out, err = _gather("present", c, ti, _dev(first), B * N)
    assert code == 0 and err == 0
    _assert_scalars(out.host, sc)
    b1 = r0 // N
    part = wr.gather_ref(slots, idx[b1:], geo)
    want_obs = part["obs"].swapaxes(1, 2).reshape(-1, W, 6, 9, 9)[r0 - b1 * N:]
    assert np.array_equal(out.host("obs", slice(r0, None)), _u16(want_obs))
    assert np.array_equal(out.host("hidden", slice(r0, None)), _u16(part["hidden"][r0 - b1 * N:]))
    assert out.guards_intact()
