"""CPU: the packed observation / comm-mask formats of the compact replay store (include/mapf_b200.h, DESIGN.md §3), the
bytes per stored transition of both layouts, and the one-hidden-vector-per-transition rule of the compact store."""
import numpy as np
import pytest

from mapf_rl_b200 import packed
from mapf_rl_b200.replay import ReplayStore


@pytest.mark.parametrize("n", [1, 6, 31, 32, 33, 64, 128])
def test_obs_pack_is_packbits_little_padded(n):
    rng = np.random.default_rng(n)
    obs = rng.random((3, n, 6, 9, 9)) < 0.4
    bits = packed.pack_obs(obs)
    assert bits.shape == (3, n, 64) and bits.dtype == np.uint8
    ref = np.packbits(obs.reshape(3, n, 486), axis=-1, bitorder="little")
    assert ref.shape[-1] == 61
    assert np.array_equal(bits[..., :61], ref)
    assert not bits[..., 61:].any()
    assert not (bits[..., 60] & 0xc0).any()                    # bits 486, 487 of the last data byte
    # element k = c*81 + r*9 + col is bit k & 7 of byte k >> 3
    c, r, col = 5, 8, 8
    k = c * 81 + r * 9 + col
    one = np.zeros((1, n, 6, 9, 9), dtype=bool)
    one[0, n - 1, c, r, col] = True
    b = packed.pack_obs(one)
    assert b.sum() == 1 << (k & 7) and b[0, n - 1, k >> 3] == 1 << (k & 7)
    back = packed.unpack_obs_np(bits)
    assert back.dtype == np.uint8 and np.array_equal(back, obs.astype(np.uint8))
    # the unpack ignores the pad bits
    dirty = bits.copy()
    dirty[..., 60] |= 0xc0
    dirty[..., 61:] = 0xff
    assert np.array_equal(packed.unpack_obs_np(dirty), obs.astype(np.uint8))


@pytest.mark.parametrize("n", [1, 6, 8, 31, 32, 33, 64, 128])
def test_comm_pack_round_trip(n):
    rng = np.random.default_rng(100 + n)
    mask = (rng.random((4, n, n)) < 0.3).astype(np.uint8)
    bits = packed.pack_comm(mask)
    cw = packed.comm_bytes(n)
    assert bits.shape == (4, n, cw) and cw == (n + 7) // 8
    assert np.array_equal(bits, np.packbits(mask, axis=-1, bitorder="little"))
    i, j = n - 1, n - 1
    one = np.zeros((1, n, n), dtype=np.uint8)
    one[0, i, j] = 1
    assert packed.pack_comm(one)[0, i, j >> 3] == 1 << (j & 7)     # LSB first
    if n % 8:
        assert not (bits[..., -1] >> (n % 8)).any()                  # bits j >= N are 0
    assert np.array_equal(packed.unpack_comm(bits, n), mask)


def test_bytes_per_transition_table():
    """DESIGN.md §3: observation + hidden + comm mask (+ action and reward) of one stored transition, latent 256."""
    rows = {6: (2916, 3072, 36, 6.0, 0.9), 32: (15552, 16384, 1024, 33.0, 2.7), 64: (31104, 32768, 4096, 68.0, 5.1)}
    for n, (obs, hid, comm, dense_kb, compact_kb) in rows.items():
        d = ReplayStore.bytes_per_transition(n, 256, compact=False)
        c = ReplayStore.bytes_per_transition(n, 256, compact=True)
        assert d == obs + hid + comm + 3
        assert c == n * 64 + n * ((n + 7) // 8) + 512 + 3
        assert round(d / 1000, 1) == dense_kb and round(c / 1000, 1) == compact_kb
    assert ReplayStore.bytes_per_transition(32, 256) / ReplayStore.bytes_per_transition(32, 256, compact=True) > 12


def test_single_hidden_rule():
    rng = np.random.default_rng(3)
    v = rng.standard_normal((5, 1, 16)).astype(np.float16)
    same = np.repeat(v, 6, axis=1)
    assert np.array_equal(packed.single_hidden(same), v[:, 0])
    assert packed.single_hidden(np.zeros((0, 6, 16), np.float16)).shape == (0, 16)
    bad = same.copy()
    bad[3, 4, 7] += 1
    with pytest.raises(ValueError):
        packed.single_hidden(bad)
