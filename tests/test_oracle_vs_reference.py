"""CPU: the C oracle (oracle/mapf_oracle.c) against the LIVE reference loaded through oracle/ref_loader.py
(MAPF_REFERENCE_DIR).  The tests that need the live reference are skipped where it is not installed; there the
oracle is pinned by the committed golden vectors instead (tests/test_oracle_golden.py).  The known-answer hashes
need only the committed copy of the reference's test instances and run everywhere.

Covers what the golden files cannot hold in bulk: random small grids at high occupancy (where the
swap / vertex / back-propagation logic of environment.py:335-406 actually fires), the SURVEY
Appendix-B known-answer hashes, search.compute_heuristics, buffer.SumTree and LocalBuffer.finish.
"""
import hashlib

import numpy as np
import pytest

from helpers import RANDOM_GRID_CASES, instances, random_grid_trials, random_instance
from oracle import oracle, ref_loader

needs_reference = pytest.mark.skipif(not ref_loader.available(), reason="the reference is not installed (MAPF_REFERENCE_DIR)")


def _ref_env(m, a, g):
    env_mod = ref_loader.load_environment()
    env = env_mod.Environment()
    env.load(np.asarray(m), np.asarray(a, dtype=np.int64), np.asarray(g, dtype=np.int64))
    return env


def _ora_env(m, a, g):
    o = oracle.OracleEnv()
    o.load(m, a, g)
    return o


# SURVEY.md Appendix B: first 16 hex digits of (navi sha256, trace sha256), #collisions, sum of final pos
KNOWN = {
    (16, 0): ("8ebb82292700f231", "806ab2023c12a3b2", 214, 621),
    (16, 199): ("efb1045ff643b96b", "2f4a011bd8ba3e8c", 287, 692),
    (32, 0): ("7b9712062d32213e", "362a683e03540220", 521, 1193),
    (32, 199): ("52c30b3ce9025e05", "3cdd652f2e52bd20", 452, 1376),
    (64, 0): ("456436d55cb98130", "ff415b2df05d69e8", 1103, 2469),
    (64, 199): ("0887e555bfaf2dda", "82f7d4e2d876086a", 1143, 2511),
}


@pytest.mark.parametrize("N,k", sorted(KNOWN))
def test_known_answer_hashes_oracle(N, k):
    """The oracle alone reproduces the hashes the surveyor took from the reference (Appendix B)."""
    maps, agents, goals = instances(N)
    acts = np.random.default_rng(0).integers(0, 5, size=(64, N))
    env = _ora_env(maps[k], agents[k], goals[k])
    navi_padded = np.pad(env.navi_map, ((0, 0), (0, 0), (4, 4), (4, 4)))
    navi_sha = hashlib.sha256(navi_padded.astype(np.uint8).tobytes()).hexdigest()[:16]
    h = hashlib.sha256()
    obs, pos = env.observe()
    h.update(obs.astype(np.uint8).tobytes())
    h.update(pos.astype(np.int64).tobytes())
    coll = 0
    for s in range(64):
        (obs, pos), r, d, _ = env.step(acts[s].tolist())
        h.update(obs.astype(np.uint8).tobytes())
        h.update(pos.astype(np.int64).tobytes())
        h.update(np.asarray(r, dtype=np.float32).tobytes())
        h.update(bytes([int(d)]))
        coll += int((np.asarray(r) == -0.5).sum())
    want = KNOWN[(N, k)]
    assert (navi_sha, h.hexdigest()[:16], coll, int(pos.sum())) == want


@needs_reference
@pytest.mark.parametrize("L,N,density,seed", RANDOM_GRID_CASES)
def test_random_grids_step_observe(L, N, density, seed):
    """High-occupancy small boards: every conflict kind of environment.py:320-406 fires."""
    for trial, (m, a, g, steps) in enumerate(random_grid_trials(L, N, density, seed)):
        ref, ora = _ref_env(m, a, g), _ora_env(m, a, g)
        assert np.array_equal(ref.navi_map[:, :, 4:-4, 4:-4].astype(np.uint8), ora.navi_map)
        for s, acts in enumerate(steps.astype(np.int64)):
            (ro, rp), rr, rd, ri = ref.step(acts.tolist())
            (oo, op), orr, od, oi = ora.step(acts.tolist())
            assert np.array_equal(rp, op), (trial, s)
            assert np.array_equal(np.asarray(rr, dtype=np.float32), np.asarray(orr, dtype=np.float32)), (trial, s)
            assert bool(rd) == od and ri == oi
            assert np.array_equal(ro.astype(np.uint8), oo.astype(np.uint8)), (trial, s)


@needs_reference
def test_finish_and_step_after_done():
    """environment.py:415-419: all rewards become `finish`; the env keeps stepping after done."""
    m = np.zeros((3, 3), dtype=np.uint8)
    a, g = np.array([[0, 0], [2, 2]]), np.array([[0, 1], [2, 1]])
    ref, ora = _ref_env(m, a, g), _ora_env(m, a, g)
    for acts in ([4, 3], [0, 0], [3, 0]):
        (_, rp), rr, rd, ri = ref.step(list(acts))
        (_, op), orr, od, oi = ora.step(list(acts))
        assert np.array_equal(rp, op) and list(map(float, rr)) == list(map(float, orr)) and bool(rd) == od and ri == oi


@needs_reference
def test_distances_vs_compute_heuristics_live():
    search = ref_loader.load_module("search")
    rng = np.random.default_rng(3)
    for L, dens in ((7, 0.3), (12, 0.35), (20, 0.3)):
        m, a, g = random_instance(rng, L, 4, dens)
        dist, _ = oracle.navi(m, g.astype(np.int32))
        for i in range(4):
            h = search.compute_heuristics(m.astype(int), (int(g[i, 0]), int(g[i, 1])))
            want = np.full((L, L), 2147483647, dtype=np.int64)
            for (x, y), c in h.items():
                want[x, y] = c
            assert np.array_equal(dist[i], want)


@needs_reference
def test_sumtree_vs_buffer_py():
    buf = ref_loader.load_module("buffer")
    rng = np.random.default_rng(5)
    cap = 1 << 10
    ref, ora = buf.SumTree(cap), oracle.OracleSumTree(cap)
    for rnd in range(30):
        n = int(rng.integers(1, 300))
        idx = rng.integers(0, cap, size=n).astype(np.int64)     # duplicates on purpose
        pr = np.where(rng.random(n) < 0.1, 0.0, rng.random(n) ** 0.6)
        ref.batch_update(idx.copy(), pr.copy())
        ora.batch_update(idx.copy(), pr.copy())
        assert np.array_equal(ref.tree, ora.tree), rnd
        if ref.tree[0] > 0:
            state = np.random.get_state()
            u_probe = np.random.random_sample(64)
            np.random.set_state(state)
            ri, rp = ref.batch_sample(64)      # consumes the same 64 uniforms from the global stream
            oi, op = ora.batch_sample(64, u_probe)
            assert np.array_equal(ri, oi) and np.array_equal(rp, op), rnd


@needs_reference
def test_actor_td_vs_local_buffer_finish():
    buf = ref_loader.load_module("buffer")
    rng = np.random.default_rng(7)
    for size in (1, 2, 5, 100, 256):
        lb = buf.LocalBuffer(0, 2, 10, np.zeros((2, 6, 9, 9), dtype=bool))
        for t in range(size):
            lb.add(rng.standard_normal(5).astype(np.float32), int(rng.integers(0, 5)), float(rng.choice([-0.075, -0.5, 0, 3])),
                   np.zeros((2, 6, 9, 9), dtype=bool), np.zeros((2, 256), dtype=np.float16), np.zeros((2, 2), dtype=bool))
        rew, q, act = lb.rew_buf[:size].copy(), lb.q_buf[:size + 1].copy(), lb.act_buf[:size].copy()
        out = lb.finish()
        td_ref = out[7]
        td = oracle.actor_td(rew, q, act, capacity=256)
        assert np.array_equal(td_ref, td)
