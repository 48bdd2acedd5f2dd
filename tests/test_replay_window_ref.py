"""CPU: the window-gather restatement (tests/replay_window_ref.py) against oracle.OracleReplay, which tests/test_replay.py pins
to the live reference GlobalBuffer and to tests/golden/replay.npz.  At every window geometry the GPU gathers are tested at
(replay_window_ref.GEOMETRIES), the same store, sum tree and uniforms give the same batch, element for element."""
import numpy as np
import pytest

import replay_window_ref as wr
from oracle import oracle
from replay_cases import ring_episodes


class _Pow2Tree(oracle.OracleSumTree):
    """The reference's sum tree takes a power-of-two capacity only, and max_steps 40 or 24 times any slot count is none: the
    tree gets the next power of two.  Leaves past the store's keep priority 0 and are never sampled."""

    def __init__(self, capacity):
        super().__init__(1 << (int(capacity) - 1).bit_length())


def _filled(geo, seed, monkeypatch):
    monkeypatch.setattr(oracle, "OracleSumTree", _Pow2Tree)
    rng = np.random.default_rng(seed)
    cap, eps = ring_episodes(geo, rng)
    ora = oracle.OracleReplay(cap, max_num_agents=geo.N, max_steps=geo.S, bt_steps=geo.bt, forward_steps=geo.fwd,
                              latent_dim=geo.latent)
    ora.add(eps)
    agents = np.full(cap, geo.N)
    slots = {g: wr.slot_of(ora.obs_buf, ora.comm_mask, ora.hid_buf, ora.act_buf, ora.rew_buf, ora.done_buf, ora.size_buf,
                           agents, g, geo.S) for g in range(cap)}
    return ora, slots, rng


def _assert_sample_equals_ref(sample, ref):
    obs, action, reward, done, steps, bt_steps, hidden, comm = sample[:8]
    u16 = lambda x: np.ascontiguousarray(x, dtype=np.float16).view(np.uint16)
    assert obs.shape == ref["obs"].shape and np.array_equal(u16(obs), u16(ref["obs"]))
    assert comm.shape == ref["comm_mask"].shape and np.array_equal(comm.astype(np.uint8), ref["comm_mask"])
    assert hidden.shape == ref["hidden"].shape and np.array_equal(u16(hidden), u16(ref["hidden"]))
    assert np.array_equal(action[:, 0], ref["action"]) and np.array_equal(bt_steps, ref["bt_steps"])
    for x, k in ((reward, "reward"), (done, "done"), (steps, "steps")):
        assert np.array_equal(u16(x[:, 0]), u16(ref[k])), k
    assert not ref["bad"].any()


@pytest.mark.parametrize("geo", wr.GEOMETRIES, ids=lambda g: "x".join(map(str, g)))
def test_gather_ref_equals_oracle_replay(geo, monkeypatch):
    ora, slots, rng = _filled(geo, sum(geo), monkeypatch)
    cap, S = len(slots), geo.S
    # the tree add() left, random uniforms
    u = rng.random(64)
    sample = ora.sample_batch(64, u)
    _assert_sample_equals_ref(sample, wr.gather_ref(slots, sample[8], geo))
    # every edge step of every slot: priority 1 on those leaves only, so sample i of the stratified draw is edge leaf i
    edges = np.asarray([g * S + t for g in range(cap) for t in wr.edge_steps(slots[g].size, geo)], dtype=np.int64)
    ora.priority_tree.batch_update(np.arange(cap * S, dtype=np.int64), np.zeros(cap * S))
    ora.priority_tree.batch_update(edges.copy(), np.ones(len(edges)))
    sample = ora.sample_batch(len(edges), rng.uniform(0.05, 0.95, size=len(edges)))
    assert np.array_equal(sample[8], edges)
    _assert_sample_equals_ref(sample, wr.gather_ref(slots, edges, geo))
    sizes = {s.size for s in slots.values()}
    assert 1 in sizes and S in sizes and len(edges) >= len(sizes)


def test_present_ref_rows_and_clamp():
    geo = wr.Geometry(5, 8, 2, 2, 3)
    rng = np.random.default_rng(1)
    agents = [1, 5, 3, 200]                      # above N: N rows
    slots = {}
    for g, n in enumerate(agents):
        slots[g] = wr.Slot(rng.random((9, 5, 6, 9, 9)) < 0.5, rng.random((9, 5, 5)) < 0.5,
                           rng.standard_normal((8, 5, 3)).astype(np.float16), rng.integers(0, 5, 8).astype(np.uint8),
                           rng.standard_normal(8).astype(np.float16), g % 2 == 0, 8, n)
    idx = np.asarray([3 * 8 + 7, 0, 8 + 4, 2 * 8 + 1, 0], dtype=np.int64)
    ref = wr.gather_ref(slots, idx, geo)
    obs, hidden, first, M, M_pad = wr.present_ref(ref, geo)
    assert M == 5 + 1 + 5 + 3 + 1 and M_pad == 256 and first.tolist() == [0, 5, 6, 11, 14]
    rows = [(b, a) for b, n in enumerate([5, 1, 5, 3, 1]) for a in range(n)]
    for m, (b, a) in enumerate(rows):
        assert np.array_equal(obs[m], ref["obs"][b, :, a]) and np.array_equal(hidden[m], ref["hidden"][b * 5 + a])
    assert not obs[M:].any() and not hidden[M:].any()
    short = wr.present_ref(ref, geo, out_rows=M - 3)
    assert short[0].shape[0] == M - 3 and np.array_equal(short[0], obs[:M - 3])
    assert ref["bad"].tolist() == [False] * 5 and ref["done"].tolist() == [0, 0, 0, 0, 0]
    assert ref["bt_steps"].tolist() == [2, 1, 2, 2, 1] and ref["steps"].tolist() == [1, 2, 2, 2, 2]
