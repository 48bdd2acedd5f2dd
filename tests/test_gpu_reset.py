"""GPU: the device-side instance generator (mapf_env_reset, Environment.reset / __init__ of
environment.py:100-138, 146-196) — distributional parity only (the reference's RNG stream is not reproduced,
SURVEY 8c), plus exact consistency of everything derived from a generated instance with the oracle.  Instance-by-instance
equality with a host restatement of the generator is in test_generator_ref.py."""
import numpy as np
import pytest

from oracle import oracle

pytestmark = pytest.mark.gpu


def make_env(B, N, L):
    from mapf_rl_b200 import BatchedEnvironment
    return BatchedEnvironment(B, N, L, device="cuda:0")


def state(env):
    return (env.map.cpu().numpy(), env.agents_pos.cpu().numpy().astype(np.int64), env.goals_pos.cpu().numpy().astype(np.int64),
            env.steps.cpu().numpy())


def check_instances(maps, pos, goals):
    B, N = pos.shape[:2]
    L = maps.shape[1]
    for k in range(B):
        cells = np.concatenate([pos[k], goals[k]])
        assert cells.min() >= 0 and cells.max() < L
        flat = cells[:, 0] * L + cells[:, 1]
        assert len(np.unique(flat)) == 2 * N, "starts and goals must be 2N distinct cells (environment.py:129-135)"
        assert maps[k][cells[:, 0], cells[:, 1]].sum() == 0, "starts / goals on free cells"
    # start and goal of each agent in one component (environment.py:120-135): goal-distance at the start is finite
    for k in range(min(B, 24)):
        dist, _ = oracle.navi(maps[k], goals[k].astype(np.int32))
        d = dist[np.arange(N), pos[k][:, 0], pos[k][:, 1]]
        assert (d < 2147483647).all() and (d > 0).all()


@pytest.mark.parametrize("L,N", [(40, 32), (40, 64), (80, 64), (20, 6), (10, 1), (33, 37), (120, 128)])
def test_reset_fixed_density(L, N):
    B = 256 if L <= 40 else 48
    env = make_env(B, N, L)
    env.reset(seed=7, density=0.3)
    env.check()
    maps, pos, goals, steps = state(env)
    assert (steps == 0).all()
    assert abs(maps.mean() - 0.3) < 0.01
    check_instances(maps, pos, goals)
    # everything derived on the device (padded bitmap, masked BFS) is consistent with the oracle on the same instance
    nv = env.navi_map.cpu().numpy()
    obs, _ = env.observe()
    obs = obs.cpu().numpy()
    rng = np.random.default_rng(0)
    acts = rng.integers(0, 5, size=(B, N)).astype(np.uint8)
    g_obs, g_rew, g_done = env.step(acts)
    g_obs, g_rew = g_obs.cpu().numpy(), g_rew.cpu().numpy()
    for k in range(min(B, 12)):
        o = oracle.OracleEnv()
        o.load(maps[k], pos[k], goals[k])
        assert np.array_equal(o.navi_map, nv[k])
        assert np.array_equal(o.observe()[0].astype(np.uint8), obs[k])
        (oo, op), orw, od, _ = o.step(acts[k])
        assert np.array_equal(oo.astype(np.uint8), g_obs[k])
        assert np.array_equal(np.asarray(orw, dtype=np.float32), g_rew[k])


def test_reset_triangular_density():
    """density=None -> one triangular(0, 0.33, 0.5) draw per environment (environment.py:100,156)."""
    B = 2048
    env = make_env(B, 4, 20)
    env.reset(seed=3)
    env.check()
    maps, pos, goals, _ = state(env)
    dens = maps.reshape(B, -1).mean(1)
    assert dens.max() < 0.62 and dens.min() >= 0.0
    assert abs(dens.mean() - (0 + 0.33 + 0.5) / 3) < 0.01          # mean of the triangular law
    # its variance (a^2+b^2+c^2-ab-ac-bc)/18 plus the Bernoulli sampling noise of a 400-cell map
    var_t = (0.33 ** 2 + 0.5 ** 2 - 0.33 * 0.5) / 18
    assert abs(dens.var() - (var_t + (dens * (1 - dens)).mean() / 400)) < 0.002
    check_instances(maps[:64], pos[:64], goals[:64])


def test_reset_deterministic_and_shardable():
    """Slot e of a batch reset with env_offset o draws the instance of global index o + e, whatever the batch."""
    big = make_env(64, 16, 40)
    big.reset(seed=11, density=0.3)
    m0, p0, g0, _ = state(big)
    again = make_env(64, 16, 40)
    again.reset(seed=11, density=0.3)
    m1, p1, g1, _ = state(again)
    assert np.array_equal(m0, m1) and np.array_equal(p0, p1) and np.array_equal(g0, g1)
    shard = make_env(16, 16, 40)
    shard.reset(seed=11, env_offset=32, density=0.3)
    m2, p2, g2, _ = state(shard)
    assert np.array_equal(m0[32:48], m2) and np.array_equal(p0[32:48], p2) and np.array_equal(g0[32:48], g2)
    other = make_env(16, 16, 40)
    other.reset(seed=12, env_offset=32, density=0.3)
    assert not np.array_equal(state(other)[0], m2)


def test_masked_reset_keeps_other_slots():
    env = make_env(32, 8, 20)
    env.reset(seed=1, density=0.25)
    acts = np.random.default_rng(0).integers(0, 5, size=(32, 8)).astype(np.uint8)
    env.step(acts)
    m0, p0, g0, s0 = state(env)
    nv0 = env.navi_map.cpu().numpy()
    mask = np.zeros(32, dtype=np.uint8)
    mask[[3, 17, 31]] = 1
    env.reset(mask=mask, seed=2, density=0.25)
    m1, p1, g1, s1 = state(env)
    nv1 = env.navi_map.cpu().numpy()
    keep = mask == 0
    assert np.array_equal(m0[keep], m1[keep]) and np.array_equal(p0[keep], p1[keep]) and np.array_equal(g0[keep], g1[keep])
    assert np.array_equal(nv0[keep], nv1[keep])
    assert (s1[keep] == 1).all() and (s1[~keep] == 0).all()
    assert not np.array_equal(m0[~keep], m1[~keep])
    check_instances(m1[~keep], p1[~keep], g1[~keep])   # (stepped slots may legitimately stand on other agents' goals)


def test_start_goal_uniformity_on_empty_board():
    """Empty 6x6 board, one agent: start uniform over 36 cells, goal uniform over the other 35 (environment.py:120-135)."""
    B = 8192
    env = make_env(B, 1, 6)
    env.reset(seed=5, density=0.0)
    _, pos, goals, _ = state(env)
    s = pos[:, 0, 0] * 6 + pos[:, 0, 1]
    g = goals[:, 0, 0] * 6 + goals[:, 0, 1]
    assert (s != g).all()
    cs = np.bincount(s, minlength=36)
    cg = np.bincount(g, minlength=36)
    exp = B / 36
    chi_s = ((cs - exp) ** 2 / exp).sum()
    chi_g = ((cg - exp) ** 2 / exp).sum()
    assert chi_s < 75 and chi_g < 75          # chi2(35): mean 35, p(>75) ~ 1e-4
    # start and goal are not correlated beyond "different": the offset g - s mod 36 is uniform over 1..35
    off = np.bincount((g - s) % 36, minlength=36)
    assert off[0] == 0 and ((off[1:] - B / 35) ** 2 / (B / 35)).sum() < 75


def test_full_board_and_overfull_board():
    env = make_env(8, 8, 4)           # 16 cells, 16 needed: every cell used
    env.reset(seed=0, density=0.0)
    env.check()
    m, p, g, _ = state(env)
    check_instances(m, p, g)
    env = make_env(4, 9, 4)           # 18 cells needed on a 16-cell board: 'no empty position' (environment.py:31)
    env.reset(seed=0, density=0.0)
    with pytest.raises(RuntimeError):
        env.check()


@pytest.mark.gpu
def test_generator_stream_is_pinned():
    """The instances of (seed, env_offset) are part of the contract (sharding, replay of a run): optimisations of the generator /
    BFS kernels must not move them.  Hash recorded with the build of round 2 (profiles/tools/r2_instance_hash.py)."""
    import hashlib
    h = hashlib.sha256()
    for (B, N, L, dens) in ((512, 32, 40, 0.3), (128, 64, 80, 0.3), (256, 7, 13, None), (64, 100, 120, 0.2)):
        env = make_env(B, N, L)
        env.reset(seed=5, env_offset=17, density=dens)
        env.check()
        for t in (env.map, env.agents_pos, env.goals_pos):
            h.update(t.cpu().numpy().tobytes())
    assert h.hexdigest() == "626f27b297399fc2c8df0dd88a7e374ea8ede2e1fabd5adecfee589bf2d4b65e"
