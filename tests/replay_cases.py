"""Shared builder of replay episodes for the ReplayStore / OracleReplay / live GlobalBuffer tests."""
import numpy as np


def make_episode(rng, actor_id, num_agents, size, done, latent=256, cap=256):
    """A tuple shaped like LocalBuffer.finish's return value (buffer.py:179; layout worker.py:72)."""
    obs = rng.random((size + 1, num_agents, 6, 9, 9)) < 0.2
    act = rng.integers(0, 5, size=size).astype(np.uint8)
    rew = rng.choice([-0.075, -0.5, 0.0, 3.0], size=size).astype(np.float16)
    hid = rng.standard_normal((size, num_agents, latent)).astype(np.float16)
    td = np.zeros(cap, dtype=np.float64)
    td[:size] = rng.random(size) * 2 + 1e-3
    comm = rng.random((size + 1, num_agents, num_agents)) < 0.3
    return (actor_id, num_agents, 10, obs, act, rew, hid, td, bool(done), size, comm)


# (num_agents, size, done) of the episodes added in order; capacity 4 => the 5th and 6th overwrite slots 0 and 1
EPISODES = [(6, 5, True), (3, 16, False), (6, 17, True), (2, 40, False), (4, 256, False), (6, 1, True)]
CAPACITY = 4
BATCH = 48


def ring_plan(geo, rng):
    """Episodes for a store at window geometry `geo` (replay_window_ref.Geometry) -> (capacity, [(num_agents, size, done)]
    in the order they are added).  Sizes 1, 2, bt - 1, bt, bt + 1, S - 1 and S (those in 1..S) each end up in two slots:
    once in a slot written once, once over a full episode (stale frames past its size); agent counts are random in 1..N and
    `done` alternates."""
    S, bt = geo.S, geo.bt
    sizes = sorted({s for s in (1, 2, bt - 1, bt, bt + 1, S - 1, S) if 1 <= s <= S})
    k = len(sizes)
    order = [S] * k + sizes + sizes      # the ring wraps after 2k: the last k overwrite the full episodes of slots 0..k-1
    return 2 * k, [(int(rng.integers(1, geo.N + 1)), s, i % 2 == 1) for i, s in enumerate(order)]


def ring_episodes(geo, rng):
    """ring_plan's episodes as LocalBuffer.finish tuples, the hidden rows of a transition equal (buffer.py:148)."""
    cap, plan = ring_plan(geo, rng)
    eps = []
    for k, (n, size, done) in enumerate(plan):
        ep = list(make_episode(rng, k, n, size, done, latent=geo.latent, cap=geo.S))
        ep[6] = np.repeat(ep[6][:, :1], n, axis=1)
        eps.append(tuple(ep))
    return cap, eps
