"""GPU: sized handles -- a per-environment agent count n_e and map side l_e inside one batch (the reference's curriculum,
worker.py:424-425).  Every output of a present agent on a cell inside l_e must equal what a uniform (n_e, l_e) handle
gives for the same instance and actions, and the oracle on the clipped instance; absent agents and off-map cells must
read exactly as include/mapf_b200.h specifies."""
import ctypes as C

import numpy as np
import pytest
from scipy import stats

from generator_ref import M32, generate, philox4x32_10
from helpers import greedy_actions, random_instance
from oracle import oracle

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
UNREACH = 2147483647
RCODE_RESET = 5
PURPOSE_LEVEL = 3

# (maxima N, L) -> settings (n_e, l_e): agent counts around the warp width and sides on both sides of the step kernel's
# row-word (24/25: 1 -> 2 words, 56/57: 2 -> 3) and the generator's / BFS's rows-per-lane boundaries (32/33), plus the
# maxima; (128, 120) runs the ranked-lookup step path (row words >= 4) for every slot
CASES = {
    (6, 40): [(1, 10), (6, 40), (3, 24), (6, 25), (1, 32), (2, 33), (4, 2), (6, 39)],
    (64, 40): [(1, 40), (31, 24), (32, 25), (33, 32), (64, 33), (64, 40), (33, 10)],
    (128, 120): [(1, 57), (31, 56), (32, 120), (33, 25), (128, 120), (128, 33), (64, 24)],
}


def level_index(seed, g, K):
    """Host restatement of the level draw of reset_levels_kernel: index (w K) >> 32, w = word 0 of Philox counter
    (g_lo, g_hi, PURPOSE_LEVEL, 0) under key (seed_lo, seed_hi)."""
    g = np.asarray(g, dtype=np.uint64)
    w = philox4x32_10(g & np.uint64(M32), g >> np.uint64(32), PURPOSE_LEVEL, 0, seed & M32, seed >> 32)[0]
    return ((w * np.uint64(K)) >> np.uint64(32)).astype(np.int64)


def padded_instances(rng, N, L, settings):
    """-> maps [B,L,L] with garbage outside l_e, agents / goals [B,N,2] with garbage rows >= n_e, and the clipped instances."""
    B = len(settings)
    maps = (rng.random((B, L, L)) < 0.5).astype(np.uint8)
    agents = rng.integers(0, 256, size=(B, N, 2)).astype(np.uint8)
    goals = rng.integers(0, 256, size=(B, N, 2)).astype(np.uint8)
    clipped = []
    for e, (n, l) in enumerate(settings):
        m, a, g = random_instance(rng, l, n, 0.0 if l * l < 4 * n else 0.2)
        maps[e, :l, :l] = m
        agents[e, :n], goals[e, :n] = a, g
        clipped.append((m, a, g))
    return maps, agents, goals, clipped


def make_sized(N, L, B):
    from mapf_rl_b200 import BatchedEnvironment
    env = BatchedEnvironment(B, N, L, device=DEV, sized=True)
    env.set_checks(True)
    return env


def uniform_handles(clipped, settings):
    from mapf_rl_b200 import BatchedEnvironment
    out = []
    for (m, a, g), (n, l) in zip(clipped, settings):
        u = BatchedEnvironment(1, n, l, device=DEV)
        u.set_checks(True)
        u.load(m[None], a[None], g[None])
        out.append(u)
    return out


def check_static(env, units, settings, N, L):
    """map, positions, goals, heuristic maps, distances and sizes of the sized handle against the uniform handles."""
    import torch
    st = env._get_state({"map", "pos", "goals", "navi", "steps"})
    mp, pos, gl, nv, sp = (st[k].cpu().numpy() for k in ("map", "pos", "goals", "navi", "steps"))
    dist = env.heuristic_distances().cpu().numpy()
    n_e, l_e = (x.cpu().numpy() for x in env.sizes)
    assert list(zip(n_e.tolist(), l_e.tolist())) == [tuple(s) for s in settings]
    for e, (u, (n, l)) in enumerate(zip(units, settings)):
        us = u._get_state({"map", "pos", "goals", "navi", "steps"})
        um = np.zeros((L, L), np.uint8)
        um[:l, :l] = us["map"][0].cpu().numpy()
        assert np.array_equal(mp[e], um), e                        # 0 outside l_e
        assert np.array_equal(pos[e, :n], us["pos"][0].cpu().numpy()) and (pos[e, n:] == 255).all()
        assert np.array_equal(gl[e, :n], us["goals"][0].cpu().numpy()) and (gl[e, n:] == 255).all()
        assert sp[e] == us["steps"][0].item()
        un = np.zeros((N, 4, L, L), np.uint8)
        un[:n, :, :l, :l] = us["navi"][0].cpu().numpy()
        assert np.array_equal(nv[e], un), e                        # 0 outside l_e and for absent agents
        ud = np.full((N, L, L), UNREACH, np.int32)
        ud[:n, :l, :l] = u.heuristic_distances().cpu().numpy()[0]
        assert np.array_equal(dist[e], ud), e
    torch.cuda.synchronize()


@pytest.mark.parametrize("maxima", list(CASES), ids=[f"{n}x{l}" for n, l in CASES])
def test_sized_equals_uniform_and_oracle(maxima):
    import torch
    N, L = maxima
    settings = CASES[maxima]
    B = len(settings)
    rng = np.random.default_rng(N * 1000 + L)
    maps, agents, goals, clipped = padded_instances(rng, N, L, settings)
    env = make_sized(N, L, B)
    env.load(maps, agents, goals, num_agents=[s[0] for s in settings], map_length=[s[1] for s in settings])
    units = uniform_handles(clipped, settings)
    oras = []
    for m, a, g in clipped:
        o = oracle.OracleEnv()
        o.load(m, a, g)
        oras.append(o)
    check_static(env, units, settings, N, L)
    # the oracle's distances / heuristic maps on the clipped instances
    nv = env.navi_map.cpu().numpy()
    for e, ((n, l), o) in enumerate(zip(settings, oras)):
        assert np.array_equal(nv[e, :n, :, :l, :l], o.navi_map)

    # first observation, plain and into store rows pre-filled with a ghost pattern
    obs0, pos0 = env.observe()
    store = torch.full((3 * B, N, 6, 9, 9), 0xAB, dtype=torch.uint8, device=DEV)
    rows = torch.arange(B, device=DEV, dtype=torch.int64) * 3 + 1
    env.observe(out_obs=store, obs_rows=rows)
    obs0, pos0, so = obs0.cpu().numpy(), pos0.cpu().numpy(), store[rows].cpu().numpy()
    for e, ((n, l), u, o) in enumerate(zip(settings, units, oras)):
        uo, up = (x.cpu().numpy()[0] for x in u.observe())
        for got in (obs0[e], so[e]):
            assert np.array_equal(got[:n], uo) and (got[n:] == 0).all()
        assert np.array_equal(uo, o.observe()[0].astype(np.uint8))
        assert np.array_equal(pos0[e, :n], up) and (pos0[e, n:] == 255).all()

    codes = torch.empty((B, N), dtype=torch.uint8, device=DEV)
    prev = [o.observe()[0].astype(np.uint8) for o in oras]
    for t in range(64):
        acts = rng.integers(0, 256, size=(B, N)).astype(np.uint8)   # garbage in the absent slots, including > 4
        for e, (n, _) in enumerate(settings):
            acts[e, :n] = rng.integers(0, 5, size=n) if t % 2 else greedy_actions(prev[e][None], rng, 0.2)[0]
        use_rows = t % 3 == 1
        if use_rows:
            store.fill_(0xAB)
            obs, rew, done = env.step(torch.as_tensor(acts, device=DEV), out_obs=store, obs_rows=rows, out_codes=codes)
            obs = store[rows]
        else:
            obs, rew, done = env.step(torch.as_tensor(acts, device=DEV), out_codes=codes)
        comm = env.comm_mask().cpu().numpy()
        obs, rew, done, cd = obs.cpu().numpy(), rew.cpu().numpy(), done.cpu().numpy(), codes.cpu().numpy()
        steps = env.steps.cpu().numpy()
        pos = env.agents_pos.cpu().numpy()
        for e, ((n, l), u, o) in enumerate(zip(settings, units, oras)):
            ucodes = torch.empty((1, n), dtype=torch.uint8, device=DEV)
            uo, ur, ud = (x.cpu().numpy()[0] for x in u.step(torch.as_tensor(acts[e:e + 1, :n], device=DEV), out_codes=ucodes))
            uc = u.comm_mask().cpu().numpy()[0]
            (oo, op), orw, od, _ = o.step(acts[e, :n])
            ctx = (maxima, e, t)
            assert np.array_equal(obs[e, :n], uo) and (obs[e, n:] == 0).all(), ctx
            assert np.array_equal(rew[e, :n], ur) and (rew[e, n:] == 0.0).all(), ctx
            assert np.array_equal(cd[e, :n], ucodes.cpu().numpy()[0]) and (cd[e, n:] == RCODE_RESET).all(), ctx
            assert done[e] == ud and steps[e] == u.steps.item() == t + 1, ctx
            assert np.array_equal(comm[e, :n, :n], uc) and not comm[e, n:].any() and not comm[e, :, n:].any(), ctx
            assert np.array_equal(uo, oo.astype(np.uint8)) and np.array_equal(ur, np.asarray(orw, np.float32)), ctx
            assert int(od) == ud and np.array_equal(pos[e, :n], op) and (pos[e, n:] == 255).all(), ctx
            assert np.array_equal(uc, oracle.comm_mask(op)), ctx
            prev[e] = uo
    env.check()                        # no action latched from the garbage bytes, no 'unique'
    check_static(env, units, settings, N, L)


def _sizes_state(env):
    st = env._get_state({"map", "pos", "goals", "navi"})
    n, l = env.sizes
    return {k: v.cpu().numpy() for k, v in dict(st, n=n, l=l).items()}


REF_LEVELS = [(n, l) for n in range(1, 7) for l in range(10, 41, 5)]


def test_reset_levels_draw_and_instances():
    from mapf_rl_b200 import BatchedEnvironment
    B, seed = 8192, 11
    env = make_sized(6, 40, B)
    env.reset(seed=seed, env_offset=0, levels=REF_LEVELS)
    env.check()
    s = _sizes_state(env)
    idx = level_index(seed, np.arange(B), len(REF_LEVELS))
    want = np.asarray(REF_LEVELS)[idx]
    assert np.array_equal(s["n"], want[:, 0]) and np.array_equal(s["l"], want[:, 1])
    counts = np.bincount(idx, minlength=len(REF_LEVELS))
    assert stats.chisquare(counts).pvalue > 1e-3
    # instance by instance: the uniform handle's reset at the drawn setting and the host restatement of the generator
    rng = np.random.default_rng(0)
    sample = np.unique(np.r_[0, B - 1, rng.integers(0, B, size=30)])
    for e in sample:
        n, l = REF_LEVELS[idx[e]]
        u = BatchedEnvironment(1, n, l, device=DEV)
        u.reset(seed=seed, env_offset=int(e))
        us = u._get_state({"map", "pos", "goals", "navi"})
        m, a, g, _ = generate(seed, int(e), l, n, None)
        assert np.array_equal(us["map"][0].cpu().numpy(), m) and np.array_equal(us["pos"][0].cpu().numpy(), a)
        assert np.array_equal(s["map"][e, :l, :l], m) and not s["map"][e, l:].any() and not s["map"][e, :, l:].any()
        assert np.array_equal(s["pos"][e, :n], a) and (s["pos"][e, n:] == 255).all()
        assert np.array_equal(s["goals"][e, :n], g) and (s["goals"][e, n:] == 255).all()
        assert np.array_equal(s["navi"][e, :n, :, :l, :l], us["navi"][0].cpu().numpy())
        assert not s["navi"][e, n:].any() and not s["navi"][e, :, :, l:].any() and not s["navi"][e, :, :, :, l:].any()
        u.close()
    # two handles covering halves of the batch draw what the full handle drew
    for half in (0, 1):
        h = make_sized(6, 40, B // 2)
        h.reset(seed=seed, env_offset=half * B // 2, levels=REF_LEVELS)
        hs = _sizes_state(h)
        sl = slice(half * B // 2, (half + 1) * B // 2)
        for k in ("n", "l", "map", "pos", "goals", "navi"):
            assert np.array_equal(hs[k], s[k][sl]), k
        h.close()
    # a masked reset leaves the other slots exactly as they were
    mask = (rng.random(B) < 0.5).astype(np.uint8)
    env.reset(mask=mask, seed=seed + 1, env_offset=B, levels=REF_LEVELS[:5])
    env.check()
    s2 = _sizes_state(env)
    keep = mask == 0
    for k in ("n", "l", "map", "pos", "goals", "navi"):
        assert np.array_equal(s2[k][keep], s[k][keep]), k
    idx2 = level_index(seed + 1, B + np.arange(B), 5)
    assert np.array_equal(s2["n"][~keep], np.asarray(REF_LEVELS[:5])[idx2[~keep], 0])


def test_reset_levels_latches_no_empty_position_per_slot():
    B, seed = 64, 5
    levels = [(1, 10), (4, 2)]                 # four agents on a 2x2 board cannot be placed: 'no empty position'
    idx = level_index(seed, np.arange(B), 2)
    env = make_sized(6, 40, B)
    env.reset(mask=(idx == 0).astype(np.uint8), seed=seed, env_offset=0, levels=levels, density=0.0)
    env.check()
    assert (env.sizes[1].cpu().numpy()[idx == 0] == 10).all()
    bad = np.zeros(B, np.uint8)
    bad[np.flatnonzero(idx == 1)[0]] = 1
    env.reset(mask=bad, seed=seed, env_offset=0, levels=levels, density=0.0)
    with pytest.raises(RuntimeError, match="no empty position"):
        env.check()


def test_sized_handle_errors():
    import torch
    from mapf_rl_b200 import _native
    from mapf_rl_b200._native import MapfError
    N, L, B = 6, 40, 4
    env = make_sized(N, L, B)
    lib, h, st = env._lib, env._h, env._stream()
    acts = torch.zeros((3, B, N), dtype=torch.uint8, device=DEV)
    for call, name in ((lambda: env.rollout(acts), "mapf_env_rollout"),
                       (lambda: env.set_autoreset(8), "mapf_env_set_autoreset"),
                       (lambda: env.step_host(np.zeros((B, N), np.uint8)), "mapf_env_step_host"),
                       (lambda: env.step_host_codes(np.zeros((B, N), np.uint8), torch.empty((B, N, 6, 9, 9), dtype=torch.uint8,
                                                                                            device=DEV)), "mapf_env_step_host_codes")):
        with pytest.raises(MapfError, match=name) as ei:
            call()
        assert ei.value.code == _native.MAPF_EINVAL
    # levels / sizes outside the maxima, and K < 1, are refused before any launch
    for levels in ([(7, 10)], [(1, 41)], [(0, 10)], [(1, 1)], [(5, 2)], [(1, 10), (2, 45)]):
        with pytest.raises(MapfError):
            env.reset(levels=levels)
    lv = torch.tensor([[1, 10]], dtype=torch.uint8, device=DEV)
    assert lib.mapf_env_reset_levels(h, None, 0, 0, C.c_float(-1.0), C.c_void_p(lv.data_ptr()), 0, st) == _native.MAPF_EINVAL
    rng = np.random.default_rng(1)
    maps, agents, goals, _ = padded_instances(rng, N, L, [(2, 10)] * B)
    for n, l in ((7, 10), (2, 41), (0, 10), (2, 1)):
        with pytest.raises(ValueError):
            env.load(maps, agents, goals, num_agents=[n] * B, map_length=[l] * B)
        nd = torch.full((B,), n, dtype=torch.uint8, device=DEV)
        ld = torch.full((B,), l, dtype=torch.uint8, device=DEV)
        md, ad, gd = (torch.as_tensor(x, device=DEV) for x in (maps, agents, goals))
        assert lib.mapf_env_load_sized(h, None, B, *(C.c_void_p(x.data_ptr()) for x in (md, ad, gd, nd, ld)), st) == _native.MAPF_EINVAL
    env.check()
    # rows >= n_e are ignored by the device too (garbage coordinates in them), and read back as 255
    md, ad, gd = (torch.as_tensor(x, device=DEV) for x in (maps, agents, goals))
    nd = torch.full((B,), 2, dtype=torch.uint8, device=DEV)
    ld = torch.full((B,), 10, dtype=torch.uint8, device=DEV)
    assert lib.mapf_env_load_sized(h, None, B, *(C.c_void_p(x.data_ptr()) for x in (md, ad, gd, nd, ld)), st) == _native.MAPF_OK
    env.check()
    p = env.agents_pos.cpu().numpy()
    assert np.array_equal(p[:, :2], agents[:, :2]) and (p[:, 2:] == 255).all()
    # a present agent's coordinate >= l_e: IndexError on the host, MAPF_ESTATE from the device-side validation
    bad = agents.copy()
    bad[1, 1] = (10, 3)
    with pytest.raises(IndexError):
        env.load(maps, bad, goals, num_agents=[2] * B, map_length=[10] * B)
    md, ad, gd = (torch.as_tensor(x, device=DEV) for x in (maps, bad, goals))
    assert lib.mapf_env_load_sized(h, None, B, *(C.c_void_p(x.data_ptr()) for x in (md, ad, gd, nd, ld)), st) == _native.MAPF_OK
    with pytest.raises(IndexError):
        env.check()
    # an absent agent's row is never looked at
    env.load(maps, bad, goals, num_agents=[1] * B, map_length=[10] * B)


def test_actor_with_curriculum():
    import torch
    from mapf_rl_b200 import ReplayStore
    from mapf_rl_b200.actor import BatchedActor
    from mapf_rl_b200.curriculum import Curriculum
    from mapf_rl_b200.qnet import Network
    torch.manual_seed(0)
    B, N, L, max_steps = 32, 6, 40, 16
    env = make_sized(N, L, B)
    net = Network().to(DEV).eval()
    store = ReplayStore(4 * B, max_num_agents=N, device=DEV)
    cur = Curriculum()
    for lv in [(2, 10), (1, 15), (3, 20), (6, 40)]:
        cur._add(lv)
    counted = np.arange(0, B, 2)
    log = dict(inst={}, steps=[], episodes=[])

    def on_begin(actor, ids):
        st = env._get_state({"map", "pos", "goals"})
        n_e, l_e = (x.cpu().numpy() for x in env.sizes)
        m, p, g = (st[k].cpu().numpy() for k in ("map", "pos", "goals"))
        for e in ids:
            n, l = int(n_e[e]), int(l_e[e])
            log["inst"][int(e)] = (m[e, :l, :l].copy(), p[e, :n].copy(), g[e, :n].copy(), len(log["steps"]), n, l)

    def on_step(actor, a8, rewards, done):
        log["steps"].append((a8.cpu().numpy(), rewards.cpu().numpy(), done.cpu().numpy()))

    def on_episode(actor, ids, slots, sizes, dones, td):
        for k, e in enumerate(ids):
            log["episodes"].append(dict(env=int(e), slot=int(slots[k]), size=int(sizes[k]), done=bool(dones[k]),
                                        inst=log["inst"][int(e)]))

    actor = BatchedActor(env, net, store, epsilon=0.3, seed=2, density=0.2, max_steps=max_steps, on_step=on_step,
                         on_episode=on_episode, on_begin=on_begin, curriculum=cur, curriculum_envs=counted)
    actor.run(48)
    env.check()
    S = store.max_steps
    obs_buf, comm_buf = store.obs_buf.cpu().numpy(), store.comm_mask.cpu().numpy()
    live = {}
    for ep in log["episodes"]:
        live[ep["slot"]] = ep
    running = {int(x) for x in actor._slot_host}
    live = {s: ep for s, ep in live.items() if s not in running}
    assert len({ep["inst"][4:] for ep in log["episodes"]}) >= 3          # several settings were drawn
    for slot, ep in live.items():
        e, size = ep["env"], ep["size"]
        m, p, g, s0, n, l = ep["inst"]
        o = oracle.OracleEnv()
        o.load(m, p.astype(np.int64), g.astype(np.int64))
        row0 = slot * (S + 1)
        assert np.array_equal(obs_buf[row0, :n], o.observe()[0].astype(np.uint8)) and not obs_buf[row0, n:].any()
        for t in range(size):
            a, r, d = log["steps"][s0 + t]
            assert np.array_equal(comm_buf[row0 + t, :n, :n], oracle.comm_mask(o.agents_pos)), (slot, t)
            assert not comm_buf[row0 + t, n:].any() and not comm_buf[row0 + t, :, n:].any()
            (oo, op), orw, od, _ = o.step(a[e, :n])
            assert np.array_equal(obs_buf[row0 + t + 1, :n], oo.astype(np.uint8)), (slot, t)
            assert not obs_buf[row0 + t + 1, n:].any(), (slot, t)
            assert np.array_equal(np.asarray(orw, dtype=np.float32), r[e, :n]) and (r[e, n:] == 0).all()
            assert int(od) == d[e]
    # the curriculum saw exactly the finished episodes of the counted environments, per setting and in order
    want = {}
    for ep in log["episodes"]:
        if ep["env"] in set(counted.tolist()):
            want.setdefault(ep["inst"][4:], []).append(ep["done"])
    got = {k: list(v) for k, v in cur.stat_dict.items() if len(v)}
    assert got == want
