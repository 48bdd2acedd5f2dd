"""The device instance generator (reset_env_warp) against a plain host restatement of it (tests/generator_ref.py).

CPU: the restatement's Philox against the Random123 known answers, the pinned instance stream of
test_gpu_reset.test_generator_stream_is_pinned reproduced on the host, and the restated law against the histograms
recorded from the live reference.  GPU: reset() instance by instance against the restatement -- map, starts, goals,
step counters and the heuristic maps of every generated environment -- at the side lengths where the generator's
templates change (RW = words per padded row 1 -> 4: L = 24 / 25, 56 / 57, 88 / 89; rows per lane 1 -> 4: L = 32 / 33,
64 / 65, 96 / 97), agent counts around the warp width, every density form, redrawn maps, 64-bit seeds and offsets and
masked resets."""
import hashlib

import numpy as np
import pytest

from generator_ref import GeneratorFailed, generate, generate_batch, philox4x32_10
from helpers import GEN_CONFIGS, generator_stats, golden, histograms_agree

PINNED_CONFIGS = ((512, 32, 40, 0.3), (128, 64, 80, 0.3), (256, 7, 13, None), (64, 100, 120, 0.2))
PINNED_HASH = "626f27b297399fc2c8df0dd88a7e374ea8ede2e1fabd5adecfee589bf2d4b65e"


@pytest.mark.parametrize("counter,key,expect", [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0), (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_philox_known_answers(counter, key, expect):
    assert tuple(int(w) for w in philox4x32_10(*counter, *key)) == expect


def test_restatement_reproduces_pinned_stream():
    """The same bytes test_generator_stream_is_pinned hashes from the device: seed 5, env_offset 17."""
    h = hashlib.sha256()
    for B, N, L, dens in PINNED_CONFIGS:
        maps, starts, goals, _ = generate_batch(5, 17, B, L, N, dens)
        for a in (maps, starts, goals):
            h.update(np.ascontiguousarray(a).tobytes())
    assert h.hexdigest() == PINNED_HASH


@pytest.mark.parametrize("L,N", GEN_CONFIGS)
def test_restated_law_matches_reference_histograms(L, N):
    """The restated generator (triangular density) draws the reference's distribution: the same two-sample chi-square
    against the live reference's histograms as test_generator_fidelity."""
    maps, starts, goals, _ = generate_batch(77 + L, 0, 3000, L, N, None)
    st = generator_stats(maps, starts, goals)
    for name, h in st.items():
        p = histograms_agree(h, golden("generator_stats.npz")[f"{name}_{L}_{N}"])
        assert p > 1e-4, f"{name} histogram differs from the reference generator at {L}x{L}/{N} agents (p = {p:.2e})"


def test_restatement_raises_without_free_cells():
    with pytest.raises(GeneratorFailed):
        generate(0, 0, 8, 2, 1.0)
    with pytest.raises(GeneratorFailed):
        generate(0, 0, 8, 2, float(np.nextafter(np.float32(1), np.float32(0))))


# ---------------------------------------------------------------------------------------------------- GPU
SIDES = [2, 3, 24, 25, 32, 33, 56, 57, 64, 65, 88, 89, 96, 97, 120]
AGENTS = [1, 31, 32, 33, 64, 97, 128]
DENSITIES = [0.0, 0.3, 0.5, None]


def batch_size(L):
    return 65 if L <= 3 else (33 if L <= 33 else (17 if L <= 65 else 5))   # odd: the last block of 4 warps is ragged


def fits(L, N):
    return N == 1 or 8 * N <= L * L


def reset_matches_restatement(env, seed, env_offset, density, slots=None, tag=""):
    """Slots `slots` (default all) of `env` hold instance env_offset + e of `seed` as restated, with steps 0 and the oracle's
    heuristic maps of the restated instance.  -> the restatement's attempt counts."""
    from oracle import oracle
    B, N, L = env.num_envs, env.num_agents, env.map_length
    slots = np.arange(B) if slots is None else np.asarray(slots)
    maps, starts, goals, steps = (x.cpu().numpy() for x in (env.map, env.agents_pos, env.goals_pos, env.steps))
    ref = [generate(seed, env_offset + int(e), L, N, density) for e in slots]
    r_maps = np.stack([r[0] for r in ref])
    r_goals = np.stack([r[2] for r in ref])
    for q, e in enumerate(slots):
        where = f"{tag} L={L} N={N} density={density} seed={seed} g={env_offset + int(e)} (slot {e})"
        assert np.array_equal(maps[e], r_maps[q]), "map differs: " + where
        assert np.array_equal(starts[e], ref[q][1]), "starts differ: " + where
        assert np.array_equal(goals[e], r_goals[q]), "goals differ: " + where
        assert steps[e] == 0, where
    import torch
    navi = env.navi_map[torch.as_tensor(slots, device=env.device)].cpu().numpy()
    r_navi = oracle.navi_batch(r_maps, r_goals)
    for q, e in enumerate(slots):
        assert np.array_equal(navi[q], r_navi[q]), f"heuristic maps differ: {tag} L={L} N={N} density={density} slot {e}"
    return np.array([r[3] for r in ref])


def make_env(B, N, L):
    from mapf_rl_b200 import BatchedEnvironment
    return BatchedEnvironment(B, N, L, device="cuda:0")


@pytest.mark.gpu
@pytest.mark.parametrize("L", SIDES)
def test_reset_matches_restatement(L):
    """Every agent count of AGENTS that fits the board, every density form, one reset each (distinct instance ranges)."""
    B = batch_size(L)
    for N in (n for n in AGENTS if fits(L, n)):
        env = make_env(B, N, L)
        for k, dens in enumerate(DENSITIES):
            off = 1000 * k + N
            env.reset(seed=L, env_offset=off, density=dens)
            env.check()
            reset_matches_restatement(env, L, off, dens)
        env.close()


@pytest.mark.gpu
def test_reset_redrawn_maps_match_restatement():
    """Small dense boards: maps without an eligible cell left for some agent are redrawn (attempt + 1)."""
    redrawn = 0
    for L, N, dens in ((2, 1, 0.5), (3, 2, 0.4), (4, 3, 0.35), (5, 4, 0.45), (6, 8, 0.4), (8, 12, None), (7, 6, 0.5)):
        env = make_env(64, N, L)
        env.reset(seed=9, env_offset=L * 100, density=dens)
        env.check()
        redrawn += int((reset_matches_restatement(env, 9, L * 100, dens) > 0).sum())
        env.close()
    assert redrawn >= 20, redrawn


@pytest.mark.gpu
@pytest.mark.parametrize("seed,offset", [((1 << 40) + 77, (1 << 32) - 7), (3, 3 * (1 << 32) + 11), ((1 << 64) - 1, (1 << 63))])
def test_reset_64bit_seed_and_offset(seed, offset):
    """Both halves of the key and of the instance counter are used (the first case crosses the low word's wrap)."""
    env = make_env(18, 33, 40)
    for dens in (0.3, None):
        env.reset(seed=seed, env_offset=offset, density=dens)
        env.check()
        reset_matches_restatement(env, seed, offset, dens)


@pytest.mark.gpu
def test_masked_reset_matches_restatement():
    """Masked slot e draws instance env_offset + e; the others keep their instance and their stepped state."""
    B, N, L = 41, 16, 33
    env = make_env(B, N, L)
    env.reset(seed=1, env_offset=0, density=0.3)
    env.check()
    env.step(np.random.default_rng(0).integers(0, 5, size=(B, N)).astype(np.uint8))
    before = [x.cpu().numpy() for x in (env.map, env.agents_pos, env.goals_pos, env.steps, env.navi_map)]
    slots = np.array([0, 3, 4, 31, 32, 40])
    mask = np.zeros(B, dtype=np.uint8)
    mask[slots] = 1
    env.reset(mask=mask, seed=2, env_offset=500, density=None)
    env.check()
    reset_matches_restatement(env, 2, 500, None, slots=slots, tag="masked")
    after = [x.cpu().numpy() for x in (env.map, env.agents_pos, env.goals_pos, env.steps, env.navi_map)]
    keep = mask == 0
    for a, b in zip(before, after):
        assert np.array_equal(a[keep], b[keep])
    assert (after[3][keep] == 1).all()
    for e in np.flatnonzero(keep)[:4]:
        m, _, g, _ = generate(1, int(e), L, N, 0.3)
        assert np.array_equal(after[0][e], m) and np.array_equal(after[2][e], g)


@pytest.mark.gpu
def test_reset_without_free_cells_raises():
    """density 1 is refused up front; the largest float below 1 leaves no free cell pair in 256 attempts and latches
    'no empty position', as the restatement raises."""
    from mapf_rl_b200 import _native
    env = make_env(4, 2, 8)
    with pytest.raises(_native.MapfError):
        env.reset(seed=0, density=1.0)
    with pytest.raises(GeneratorFailed):
        generate(0, 0, 8, 2, 1.0)
    below_one = float(np.nextafter(np.float32(1), np.float32(0)))
    env.reset(seed=0, env_offset=0, density=below_one)
    with pytest.raises(RuntimeError, match="no empty position"):
        env.check()
    with pytest.raises(GeneratorFailed):
        generate(0, 0, 8, 2, below_one)
    env.reset(seed=0, env_offset=0, density=0.2)      # the latch was cleared by check(): the handle is usable again
    env.check()
    reset_matches_restatement(env, 0, 0, 0.2)
