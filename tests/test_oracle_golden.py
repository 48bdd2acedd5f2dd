"""CPU: the C oracle (oracle/mapf_oracle.c) against the golden vectors generated from the live
reference (tests/golden/make_golden.py).  This is what pins the oracle on a box without /root/reference."""
import hashlib

import numpy as np
import pytest

from helpers import RANDOM_GRID_CASES, golden, instances
from oracle import oracle


def sha8(b):
    return np.frombuffer(hashlib.sha256(b).digest()[:8], dtype=np.uint64)[0]


@pytest.mark.parametrize("N", [16, 32, 64])
@pytest.mark.parametrize("stream", ["U", "G"])
def test_traces(N, stream):
    z = golden("traces.npz")
    maps, agents, goals = instances(N)
    pre = f"n{N}_{stream}_"
    for q, k in enumerate(z[pre + "instances"]):
        env = oracle.OracleEnv()
        env.load(maps[k], agents[k], goals[k])
        obs, pos = env.observe()
        assert np.array_equal(pos, z[pre + "pos"][q, 0])
        assert sha8(obs.astype(np.uint8).tobytes()) == z[pre + "obs_sha8"][q, 0]
        for s in range(z[pre + "actions"].shape[1]):
            (obs, pos), r, d, info = env.step(z[pre + "actions"][q, s].tolist())
            assert info == {"step": s}
            assert np.array_equal(pos, z[pre + "pos"][q, s + 1]), (k, s)
            assert np.array_equal(np.asarray(r, dtype=np.float32), z[pre + "rewards"][q, s]), (k, s)
            assert int(d) == z[pre + "done"][q, s]
            assert sha8(obs.astype(np.uint8).tobytes()) == z[pre + "obs_sha8"][q, s + 1], (k, s)
        last = np.unpackbits(z[pre + "obs_last_packed"][q])[: N * 486].reshape(N, 6, 9, 9)
        assert np.array_equal(obs.astype(np.uint8), last)


@pytest.mark.parametrize("N", [16, 32, 64])
def test_navi_all_instances(N):
    z = golden("navi.npz")
    maps, agents, goals = instances(N)
    for k in range(200):
        _, nv = oracle.navi(maps[k], goals[k].astype(np.int32))
        got = np.frombuffer(hashlib.sha256(nv.tobytes()).digest(), dtype=np.uint8)
        assert np.array_equal(got, z[f"navi{N}_sha256"][k]), k
        if f"navi{N}_{k}_packed" in z:
            full = np.unpackbits(z[f"navi{N}_{k}_packed"])[: N * 4 * 1600].reshape(N, 4, 40, 40)
            assert np.array_equal(nv, full)


def test_distances_vs_compute_heuristics():
    z = golden("navi.npz")
    maps, agents, goals = instances(32)
    for k in (0, 199):
        dist, _ = oracle.navi(maps[k], goals[k].astype(np.int32))
        assert np.array_equal(dist, z[f"dist32_{k}"])


def test_crafted_cases():
    z = golden("crafted.npz")
    for name in z["names"]:
        env = oracle.OracleEnv()
        env.load(z[f"{name}_map"], z[f"{name}_agents"], z[f"{name}_goals"])
        (obs, pos), r, d, info = env.step(z[f"{name}_actions"].tolist())
        assert np.array_equal(pos, z[f"{name}_pos"]), name
        assert np.array_equal(np.asarray(r, dtype=np.float32), z[f"{name}_rewards"]), name
        assert int(d) == z[f"{name}_done"], name
        assert np.array_equal(obs.astype(np.uint8), z[f"{name}_obs"]), name
        (obs, pos), r, d, info = env.step([0] * len(pos))
        assert np.array_equal(np.asarray(r, dtype=np.float32), z[f"{name}_rewards2"]), name
        assert int(d) == z[f"{name}_done2"] and info["step"] == z[f"{name}_info2"]


def test_sumtree_rounds():
    z = golden("per.npz")
    tree = oracle.OracleSumTree(int(z["capacity"]))
    for rd in range(int(z["rounds"])):
        idx = z[f"upd_idx_{rd}"].copy()
        tree.batch_update(idx, z[f"upd_prio_{rd}"])
        assert np.array_equal(idx, z[f"upd_idx_{rd}"] + tree.capacity - 1)  # buffer.py:96 in-place mutation
        got = np.frombuffer(hashlib.sha256(tree.tree.tobytes()).digest(), dtype=np.uint8)
        assert np.array_equal(got, z[f"tree_sha_{rd}"]), rd
        sidx, sprio = tree.batch_sample(len(z[f"smp_u_{rd}"]), z[f"smp_u_{rd}"])
        assert np.array_equal(sidx, z[f"smp_idx_{rd}"]), rd
        assert np.array_equal(sprio, z[f"smp_prio_{rd}"]), rd
    assert np.array_equal(tree.tree, z["tree_final"])
    assert abs(tree.tree[-tree.capacity:].sum() - tree.tree[0]) < 0.1  # buffer.py:105


def test_actor_td():
    z = golden("per.npz")
    for case in range(5):
        td = oracle.actor_td(z[f"td_rew_{case}"], z[f"td_q_{case}"], z[f"td_act_{case}"])
        assert np.array_equal(td, z[f"td_out_{case}"]), case


@pytest.mark.parametrize("case", range(len(RANDOM_GRID_CASES)))
def test_random_grids_recorded(case):
    """The oracle on the high-occupancy random boards of helpers.RANDOM_GRID_CASES against its recorded trajectories
    (tests/golden/make_random_grids.py; test_oracle_vs_reference.py checks the same boards against the live reference)."""
    z = golden("random_grids.npz")
    pre = f"c{case}_"
    for t in range(z[pre + "map"].shape[0]):
        env = oracle.OracleEnv()
        env.load(z[pre + "map"][t], z[pre + "agents"][t], z[pre + "goals"][t])
        assert sha8(np.ascontiguousarray(env.navi_map, dtype=np.uint8).tobytes()) == z[pre + "navi_sha8"][t]
        obs, pos = env.observe()
        assert np.array_equal(pos, z[pre + "pos"][t, 0])
        assert sha8(obs.astype(np.uint8).tobytes()) == z[pre + "obs_sha8"][t, 0]
        for s, acts in enumerate(z[pre + "actions"][t]):
            (obs, pos), r, d, info = env.step(acts.tolist())
            assert info == {"step": s}
            assert np.array_equal(pos, z[pre + "pos"][t, s + 1]), (t, s)
            assert np.array_equal(np.asarray(r, dtype=np.float32), z[pre + "rewards"][t, s]), (t, s)
            assert int(d) == z[pre + "done"][t, s], (t, s)
            assert sha8(obs.astype(np.uint8).tobytes()) == z[pre + "obs_sha8"][t, s + 1], (t, s)
        assert np.array_equal(np.packbits(obs.astype(np.uint8).ravel()), z[pre + "obs_last_packed"][t])
