"""GPU: the compact replay store.  Packed step / observe / comm mask equal np.packbits of the dense entry points (padding
included) with the same step results; mapf_obs_unpack equals the numpy restatement; the compact gather returns bit-identical
batches to the dense gather for the same logical store; a dense-store and a compact-store BatchedActor driven by the same
deterministic policy leave the same store behind; and the real Network trains from a compact store."""
import ctypes as C

import numpy as np
import pytest

from helpers import greedy_actions, random_instance
from mapf_rl_b200 import packed

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# (N, L): one to four agents per lane on every map-width class; L * L leaves room for the agents
STEP_CASES = [(n, l) for n in (1, 6, 31, 32, 33, 64, 128) for l in (10, 40, 80, 120) if l * l >= 2 * n]


def _load_pair(N, L, B, seed):
    from mapf_rl_b200 import BatchedEnvironment
    rng = np.random.default_rng(seed)
    dens = 0.3 if L * L * 0.7 >= 3 * N else 0.05
    inst = [random_instance(rng, L, N, dens) for _ in range(B)]
    m, a, g = (np.stack(x) for x in zip(*inst))
    envs = []
    for _ in range(2):
        e = BatchedEnvironment(B, N, L, device=DEV)
        e.set_checks(True)
        e.load(m, a, g)
        envs.append(e)
    return envs, rng


@pytest.mark.parametrize("N,L", STEP_CASES)
def test_packed_step_and_observe_equal_packed_dense(N, L):
    import torch
    B, T = 12, 24
    (dense, pk), rng = _load_pair(N, L, B, 7 * N + L)
    F = 3 * B
    bits = torch.full((F, N, 64), 0xAB, dtype=torch.uint8, device=DEV)
    obs, pos = dense.observe()
    _, ppos = pk.observe(out_bits=bits)
    assert np.array_equal(bits[:B].cpu().numpy(), packed.pack_obs(obs.cpu().numpy()))
    assert torch.equal(pos, ppos)
    prev = obs.cpu().numpy()
    codes_d = torch.empty((B, N), dtype=torch.uint8, device=DEV)
    codes_p = torch.empty_like(codes_d)
    for t in range(T):
        acts = rng.integers(0, 5, size=(B, N)).astype(np.uint8) if t % 2 else greedy_actions(prev, rng, 0.1)
        a = torch.as_tensor(acts, device=DEV)
        rows = None
        if t % 3:   # row-addressed into a larger buffer, in a scrambled order
            rows = torch.as_tensor(rng.permutation(F)[:B], dtype=torch.int64, device=DEV)
        bits.fill_(0xAB)                                   # every byte of a written frame, pads included, must be rewritten
        o_d, r_d, d_d = dense.step(a, out_codes=codes_d)
        o_p, r_p, d_p = pk.step(a, out_bits=bits, obs_rows=rows, out_codes=codes_p)
        assert o_p is bits
        got = bits.cpu().numpy()
        got = got[rows.cpu().numpy()] if rows is not None else got[:B]
        want = packed.pack_obs(o_d.cpu().numpy())
        assert np.array_equal(got, want), (N, L, t)
        assert torch.equal(r_d, r_p) and torch.equal(d_d, d_p) and torch.equal(codes_d, codes_p)
        assert torch.equal(dense._steps, pk._steps) and torch.equal(dense.agents_pos, pk.agents_pos)
        prev = o_d.cpu().numpy()
    # frames nobody wrote keep the fill: the kernel writes exactly its rows
    rows = torch.as_tensor(np.arange(B)[::-1].copy() * 2 + 1, dtype=torch.int64, device=DEV)
    bits.fill_(0xAB)
    pk.observe(out_bits=bits, obs_rows=rows)
    g = bits.cpu().numpy()
    assert np.array_equal(g[rows.cpu().numpy()], packed.pack_obs(dense.observe()[0].cpu().numpy()))
    untouched = np.setdiff1d(np.arange(F), rows.cpu().numpy())
    assert (g[untouched] == 0xAB).all()
    dense.check()
    pk.check()


@pytest.mark.parametrize("N,L", [(6, 40), (33, 80), (64, 120)])
def test_packed_sized_absent_rows_zero_present_match_uniform(N, L):
    import torch
    from test_gpu_sized import make_sized, padded_instances, uniform_handles
    rng = np.random.default_rng(N + L)
    settings = [(1, 2), (N, L), (max(1, N // 3), L // 2), (N, 10), (2, L), (max(1, N - 1), L - 3)]
    B = len(settings)
    maps, agents, goals, clipped = padded_instances(rng, N, L, settings)
    env = make_sized(N, L, B)
    env.load(maps, agents, goals, num_agents=[s[0] for s in settings], map_length=[s[1] for s in settings])
    units = uniform_handles(clipped, settings)
    bits = torch.full((B, N, 64), 0xAB, dtype=torch.uint8, device=DEV)

    def check(tag):
        got = bits.cpu().numpy()
        for e, (n, l) in enumerate(settings):
            uo = units[e].observe()[0].cpu().numpy()
            assert np.array_equal(got[e, :n], packed.pack_obs(uo)[0]), (tag, e)
            assert not got[e, n:].any(), (tag, e)

    env.observe(out_bits=bits)
    check("observe")
    prev = [u.observe()[0].cpu().numpy() for u in units]
    codes = torch.empty((B, N), dtype=torch.uint8, device=DEV)
    for t in range(16):
        acts = rng.integers(0, 5, size=(B, N)).astype(np.uint8)
        for e, (n, l) in enumerate(settings):
            if t % 2 == 0:
                acts[e, :n] = greedy_actions(prev[e], rng, 0.2)[0]
        bits.fill_(0xAB)
        _, rew, done = env.step(torch.as_tensor(acts, device=DEV), out_bits=bits, out_codes=codes)
        rew, done, codes_h = rew.cpu().numpy(), done.cpu().numpy(), codes.cpu().numpy()
        for e, (n, l) in enumerate(settings):
            uo, ur, ud = units[e].step(acts[e:e + 1, :n])
            prev[e] = uo.cpu().numpy()
            assert np.array_equal(rew[e, :n], ur[0].cpu().numpy()) and (rew[e, n:] == 0).all()
            assert (codes_h[e, n:] == 5).all() and done[e] == int(ud[0])
        check(t)
    env.check()


def test_packed_comm_mask_uniform_and_sized():
    import torch
    from mapf_rl_b200 import BatchedEnvironment, _native
    from test_gpu_sized import make_sized, padded_instances
    rng = np.random.default_rng(11)
    for N, L in ((6, 10), (13, 12), (32, 40), (64, 40), (128, 80)):
        env = BatchedEnvironment(24, N, L, device=DEV)
        env.reset(seed=N, env_offset=0, density=0.1)
        env.check()
        CW = (N + 7) // 8
        for k in (1, 2, 3):
            dense = env.comm_mask(k)
            bits = torch.full((50, N, CW), 0xAB, dtype=torch.uint8, device=DEV)
            rows = torch.as_tensor(rng.permutation(50)[:24], dtype=torch.int64, device=DEV)
            d2 = env.comm_mask(k, out_bits=bits, rows=rows)
            assert torch.equal(d2, dense)
            assert np.array_equal(bits.cpu().numpy()[rows.cpu().numpy()], packed.pack_comm(dense.cpu().numpy())), (N, k)
            # packed rows only (no dense output), consecutive
            b2 = torch.full((24, N, CW), 0xAB, dtype=torch.uint8, device=DEV)
            _native.check(env._lib.mapf_env_comm_mask_packed(env._h, k, None, C.c_void_p(b2.data_ptr()), None, env._stream()))
            assert torch.equal(b2, bits[rows])
    N, L = 33, 40
    settings = [(1, 10), (33, 40), (9, 20), (32, 40), (17, 12)]
    maps, agents, goals, _ = padded_instances(rng, N, L, settings)
    env = make_sized(N, L, len(settings))
    env.load(maps, agents, goals, num_agents=[s[0] for s in settings], map_length=[s[1] for s in settings])
    bits = torch.full((len(settings), N, 5), 0xAB, dtype=torch.uint8, device=DEV)
    d2 = env.comm_mask(3, out_bits=bits)
    assert torch.equal(d2, env.comm_mask(3))
    assert np.array_equal(bits.cpu().numpy(), packed.pack_comm(d2.cpu().numpy()))
    for e, (n, l) in enumerate(settings):
        assert not bits[e, n:].any()


@pytest.mark.parametrize("N", [1, 6, 31, 32, 33, 128])
def test_obs_unpack_matches_numpy(N):
    import torch
    rng = np.random.default_rng(N)
    F = 40
    raw = rng.integers(0, 256, size=(F, N, 64)).astype(np.uint8)    # pad bits set: the unpack ignores them
    bits = torch.as_tensor(raw, device=DEV)
    want = packed.unpack_obs_np(raw)
    rows = torch.as_tensor(rng.integers(0, F, size=17), dtype=torch.int64, device=DEV)
    for dt in (torch.uint8, torch.float16, torch.bfloat16):
        full = packed.unpack_obs(bits, dtype=dt)
        assert full.dtype == dt and tuple(full.shape) == (F, N, 6, 9, 9)
        assert np.array_equal(full.float().cpu().numpy(), want.astype(np.float32)), dt
        sel = packed.unpack_obs(bits, rows, dtype=dt)
        assert np.array_equal(sel.float().cpu().numpy(), want[rows.cpu().numpy()].astype(np.float32)), dt


def _store_pair(N, latent, cap, S, rng, sizes, dones):
    """A dense and a compact ReplayStore with the same logical contents (hidden rows of a transition equal)."""
    import torch
    from mapf_rl_b200 import ReplayStore
    kw = dict(max_num_agents=N, device=DEV, max_steps=S, latent_dim=latent)
    d, c = ReplayStore(cap, **kw), ReplayStore(cap, compact=True, **kw)
    R = (S + 1) * cap
    obs = rng.random((R, N, 6, 9, 9)) < 0.3
    comm = rng.random((R, N, N)) < 0.3
    hid = rng.standard_normal((S * cap, latent)).astype(np.float16)
    d.obs_buf.copy_(torch.as_tensor(obs.astype(np.uint8)))
    d.comm_mask.copy_(torch.as_tensor(comm.astype(np.uint8)))
    d.hid_buf.copy_(torch.as_tensor(hid)[:, None, :].expand(S * cap, N, latent))
    c.obs_bits.copy_(torch.as_tensor(packed.pack_obs(obs)))
    c.comm_bits.copy_(torch.as_tensor(packed.pack_comm(comm)))
    c.hid_buf.copy_(torch.as_tensor(hid))
    act = torch.as_tensor(rng.integers(0, 5, size=S * cap).astype(np.uint8))
    rew = torch.as_tensor(rng.choice([-0.075, -0.5, 0.0, 3.0], size=S * cap).astype(np.float16))
    for s in (d, c):
        s.act_buf.copy_(act)
        s.rew_buf.copy_(rew)
        s.size_buf.copy_(torch.as_tensor(np.asarray(sizes, dtype=np.int32)))
        s.done_buf.copy_(torch.as_tensor(np.asarray(dones, dtype=np.uint8)))
    return d, c


@pytest.mark.parametrize("N,latent", [(6, 256), (13, 256), (32, 256), (33, 12), (8, 20)])
def test_compact_gather_equals_dense_gather(N, latent):
    import torch
    rng = np.random.default_rng(N * 1000 + latent)
    cap, S = 8, 32                          # the sum tree needs cap * S to be a power of two
    sizes = [S, 1, 17, 3, S, 25, 16, 31]    # full, one-step and short episodes
    dones = [0, 1, 1, 0, 1, 0, 1, 0]
    d, c = _store_pair(N, latent, cap, S, rng, sizes, dones)
    g = np.arange(cap)
    idx = []
    for slot in g:
        for t in sorted({0, 1, d.bt_steps - 1, d.bt_steps, sizes[slot] - 2, sizes[slot] - 1}):
            if 0 <= t < sizes[slot]:
                idx.append(slot * S + t)
    idx += list(rng.integers(0, cap * S, size=40))   # includes leaves beyond their episode's size
    idx = torch.as_tensor(np.asarray(idx, dtype=np.int64), device=DEV)
    od, oc = d.gather(idx), c.gather(idx)
    for k in od:
        assert od[k].dtype == oc[k].dtype and od[k].shape == oc[k].shape, k
        assert torch.equal(od[k].view(torch.uint8) if od[k].is_floating_point() else od[k],
                           oc[k].view(torch.uint8) if oc[k].is_floating_point() else oc[k]), k
    assert int(d._err.item()) == int(c._err.item()) == 1             # some leaves lie beyond their episode
    # only leaves inside their episodes: no latch on either
    d._err.zero_(), c._err.zero_()
    ok = idx[:len(idx) - 40]
    od, oc = d.gather(ok), c.gather(ok)
    assert all(torch.equal(od[k], oc[k]) for k in od)
    assert int(d._err.item()) == int(c._err.item()) == 0
    # sample_batch from equal trees with the same uniforms
    leaves = np.concatenate([np.arange(s * S, s * S + sizes[s]) for s in g])
    pr = rng.random(len(leaves)) + 0.1
    for s in (d, c):
        s.priority_tree.batch_update(leaves.copy(), pr.copy())
    u = rng.random(64)
    bd, bc = d.sample_batch(64, uniforms=u), c.sample_batch(64, uniforms=u)
    for x, y in zip(bd, bc):
        if isinstance(x, np.ndarray):
            assert np.array_equal(x, y)
        elif hasattr(x, "shape"):
            assert torch.equal(x, y)
        else:
            assert x == y


def test_compact_add_packs_the_reference_tuple():
    import torch
    from replay_cases import make_episode
    from mapf_rl_b200 import ReplayStore
    rng = np.random.default_rng(5)
    N, S = 6, 32
    d = ReplayStore(4, max_num_agents=N, device=DEV, max_steps=S)
    c = ReplayStore(4, max_num_agents=N, device=DEV, max_steps=S, compact=True)
    eps = []
    for n, size, done in [(6, 5, True), (6, 32, False), (6, 17, True)]:
        ep = list(make_episode(rng, 0, n, size, done, latent=256, cap=S))
        ep[6] = np.repeat(ep[6][:, :1], n, axis=1)                # the reference's broadcast hidden rows
        eps.append(tuple(ep))
    d.add(eps)
    c.add(eps)
    assert np.array_equal(packed.unpack_obs_np(c.obs_bits.cpu().numpy()), d.obs_buf.cpu().numpy())
    assert np.array_equal(packed.unpack_comm(c.comm_bits.cpu().numpy(), N), d.comm_mask.cpu().numpy())
    assert torch.equal(d.hid_buf[:, 0], c.hid_buf) and torch.equal(d.hid_buf, c.hid_buf[:, None].expand_as(d.hid_buf))
    bad = list(make_episode(rng, 0, N, 4, False, latent=256, cap=S))     # hidden rows of a transition differ
    ptr = c.ptr
    with pytest.raises(ValueError):
        c.add([tuple(bad)])
    assert c.ptr == ptr


class _PolicyStub:
    """Actions, q and hidden as pure functions of (obs, comm): a dense-store and a compact-store actor see the same inputs
    and must make the same moves."""

    def __init__(self, latent):
        self.latent = latent

    def reset(self):
        pass

    def step(self, obs, comm, reset_mask=None):
        import torch
        B, N = obs.shape[:2]
        o = obs.reshape(B, N, -1).float()
        navi = o.reshape(B, N, 6, 9, 9)[:, :, 2:6, 4, 4]
        key = navi * (1 + torch.arange(4, device=obs.device, dtype=torch.float32)) + (o.sum(-1, keepdim=True) % 3 == 0) * 2.5
        actions = torch.where(navi.sum(-1) > 0, 1 + key.argmax(-1), torch.zeros_like(navi[..., 0], dtype=torch.int64))
        q = torch.cat([o[:, :, :4] + 0.25 * comm.float().sum(-1, keepdim=True), o[:, :, 4:5]], -1)
        hidden = o[:, :, :self.latent] * 0.5 + comm.float().sum(-1, keepdim=True) / N
        return actions, q, hidden


@pytest.mark.parametrize("curriculum", [False, True])
def test_actor_twin_dense_and_compact(curriculum):
    import torch
    from mapf_rl_b200 import BatchedEnvironment, ReplayStore
    from mapf_rl_b200.actor import BatchedActor
    from mapf_rl_b200.curriculum import Curriculum
    B, N, L, S = 16, 6, 20, 16              # 2 B slots x S steps: the sum tree needs a power of two
    latent = 32
    out = []
    for compact in (False, True):
        env = BatchedEnvironment(B, N, L, device=DEV, sized=curriculum)
        cur = None
        if curriculum:
            cur = Curriculum()
            for lv in [(2, 10), (1, 15), (4, 20), (6, 20)]:
                cur._add(lv)
        store = ReplayStore(2 * B, max_num_agents=N, device=DEV, max_steps=S, latent_dim=latent, compact=compact)
        actor = BatchedActor(env, _PolicyStub(latent), store, epsilon=0.2, seed=3, density=0.2, max_steps=S, curriculum=cur)
        actor.run(5 * S)
        env.check()
        store.priority_tree.check()
        out.append((actor, store, cur))
    (ad, d, cd), (ac, c, cc) = out
    assert ad.episodes == ac.episodes >= 3 * B and ad.episodes > 0
    assert np.array_equal(packed.unpack_obs_np(c.obs_bits.cpu().numpy()), d.obs_buf.cpu().numpy())
    assert np.array_equal(packed.unpack_comm(c.comm_bits.cpu().numpy(), N), d.comm_mask.cpu().numpy())
    assert torch.equal(d.hid_buf, c.hid_buf[:, None].expand_as(d.hid_buf))
    for k in ("act_buf", "rew_buf", "done_buf", "size_buf"):
        assert torch.equal(getattr(d, k), getattr(c, k)), k
    assert torch.equal(d.priority_tree.tree.view(torch.int64), c.priority_tree.tree.view(torch.int64))
    assert d.size == c.size and d.ptr == c.ptr
    if curriculum:
        assert {k: list(v) for k, v in cd.stat_dict.items()} == {k: list(v) for k, v in cc.stat_dict.items()}
    u = np.random.default_rng(1).random(96)
    bd, bc = d.sample_batch(96, uniforms=u), c.sample_batch(96, uniforms=u)
    for x, y in zip(bd, bc):
        if isinstance(x, np.ndarray):
            assert np.array_equal(x, y)
        elif hasattr(x, "shape"):
            assert torch.equal(x, y)
        else:
            assert x == y


def test_network_trains_from_compact_store():
    import torch
    from mapf_rl_b200 import BatchedEnvironment, ReplayStore
    from mapf_rl_b200.actor import BatchedActor
    from mapf_rl_b200.learner import BatchedLearner
    from mapf_rl_b200.qnet import Network
    torch.manual_seed(0)
    B, N, L, cap = 48, 4, 12, 16
    env = BatchedEnvironment(B, N, L, device=DEV)
    net = Network().to(DEV)
    store = ReplayStore(128, max_num_agents=N, device=DEV, max_steps=cap, compact=True)
    assert store.nbytes < ReplayStore.bytes_per_transition(N, compact=False) * 128 * cap
    actor = BatchedActor(env, net, store, epsilon=0.3, seed=1, density=0.15, max_steps=cap)
    actor.run(2 * cap + 3)
    assert actor.episodes >= 2 * B and len(store) >= 192
    learner = BatchedLearner(net, store, batch_size=64, target_update_freq=3, seed=5)
    for _ in range(4):
        stats = learner.update(want_stats=True)
        assert np.isfinite(stats["loss"])
    actor.run(3)
    env.check()
    store.priority_tree.check()
