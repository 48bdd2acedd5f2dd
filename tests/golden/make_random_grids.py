#!/usr/bin/env python
"""Writes tests/golden/random_grids.npz: the C oracle's trajectories on the high-occupancy random boards of
helpers.RANDOM_GRID_CASES (swaps, vertex conflicts, chains backing up behind a blocked agent).

Recorded from the oracle, NOT from the reference: where the reference is installed,
tests/test_oracle_vs_reference.py::test_random_grids_step_observe checks the oracle against it on exactly these boards;
tests/test_oracle_golden.py::test_random_grids_recorded keeps the oracle on these trajectories everywhere else.
Inputs (boards, actions) are stored too, so the file does not depend on numpy's random streams.

    python tests/golden/make_random_grids.py
"""
from __future__ import annotations

import hashlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.abspath(os.path.join(HERE, "..", "..")))
sys.path.insert(0, os.path.abspath(os.path.join(HERE, "..")))

from helpers import RANDOM_GRID_CASES, random_grid_trials  # noqa: E402
from oracle import oracle  # noqa: E402


def sha8(b: bytes) -> np.uint64:
    return np.frombuffer(hashlib.sha256(b).digest()[:8], dtype=np.uint64)[0]


def main():
    out = {"cases": np.array(RANDOM_GRID_CASES, dtype=np.float64)}
    for c, (L, N, density, seed) in enumerate(RANDOM_GRID_CASES):
        trials = random_grid_trials(L, N, density, seed)
        T = trials[0][3].shape[0]
        rec = {k: [] for k in ("map", "agents", "goals", "actions", "navi_sha8", "pos", "rewards", "done", "obs_sha8", "obs_last_packed")}
        for m, a, g, acts in trials:
            env = oracle.OracleEnv()
            env.load(m, a, g)
            obs, pos = env.observe()
            pos_t, rew_t, done_t, sha_t = [pos.astype(np.uint8)], [], [], [sha8(obs.astype(np.uint8).tobytes())]
            for s in range(T):
                (obs, pos), r, d, info = env.step(acts[s].tolist())
                assert info == {"step": s}
                pos_t.append(pos.astype(np.uint8))
                rew_t.append(np.asarray(r, dtype=np.float32))
                done_t.append(int(d))
                sha_t.append(sha8(obs.astype(np.uint8).tobytes()))
            rec["map"].append(m.astype(np.uint8))
            rec["agents"].append(a)
            rec["goals"].append(g)
            rec["actions"].append(acts)
            rec["navi_sha8"].append(sha8(np.ascontiguousarray(env.navi_map, dtype=np.uint8).tobytes()))
            rec["pos"].append(np.stack(pos_t))
            rec["rewards"].append(np.stack(rew_t))
            rec["done"].append(np.array(done_t, dtype=np.uint8))
            rec["obs_sha8"].append(np.array(sha_t, dtype=np.uint64))
            rec["obs_last_packed"].append(np.packbits(obs.astype(np.uint8).ravel()))
        for k, v in rec.items():
            out[f"c{c}_{k}"] = np.stack(v)
    path = os.path.join(HERE, "random_grids.npz")
    np.savez_compressed(path, **out)
    print(f"{path}: {os.path.getsize(path)} bytes")


if __name__ == "__main__":
    main()
