"""CPU: the curriculum's statistics and growth rule (GlobalBuffer.stat_dict / stats, worker.py:73-82, 205-226), and that
the Q-network gives present agents the same outputs whether or not absent agents are padded in (zero observation rows,
zero comm rows and columns) -- what makes an episode of a sized batch in the N-agent replay store equivalent to the
reference's n-agent episode."""
import numpy as np
import pytest

from mapf_rl_b200.curriculum import Curriculum


def fill(c, level, successes, total=200):
    c.record([level[0]] * total, [level[1]] * total, [True] * successes + [False] * (total - successes))


def test_starts_at_init_set():
    c = Curriculum()
    assert c.levels == [(1, 10)]
    assert c.advance() == []


def test_window_keeps_the_last_200_results():
    c = Curriculum()
    fill(c, (1, 10), 0, 1)                 # the oldest result: a failure
    fill(c, (1, 10), 180, 199)             # window full: 180 successes and the failure
    w = c.stat_dict[(1, 10)]
    assert len(w) == 200 and sum(w) == 180 and w[0] is False
    c.record([1], [10], [True])            # the 201st result drops the oldest
    assert len(w) == 200 and sum(w) == 181 and w[0] is True


@pytest.mark.parametrize("successes, grows", [(180, True), (179, False)])
def test_threshold(successes, grows):
    c = Curriculum()
    fill(c, (1, 10), successes)
    added = c.advance()
    assert (added == [(2, 10), (1, 15)]) == grows
    assert c.levels == ([(1, 10), (2, 10), (1, 15)] if grows else [(1, 10)])


def test_partial_window_does_not_grow():
    c = Curriculum()
    fill(c, (1, 10), 199, 199)
    assert c.advance() == []


def test_growth_stops_at_the_maxima_no_duplicates_insertion_order():
    c = Curriculum(max_num_agents=3, max_map_length=20)
    order = []
    for _ in range(10):
        for level in c.levels:
            fill(c, level, 200)
        added = c.advance()
        order += added
        if not added:
            break
    assert c.levels == [(1, 10)] + order
    assert len(set(c.levels)) == len(c.levels)
    assert set(c.levels) == {(n, l) for n in (1, 2, 3) for l in (10, 15, 20)}
    # first round: (1,10) -> (2,10), (1,15); second round visits them in insertion order
    assert c.levels[:5] == [(1, 10), (2, 10), (1, 15), (3, 10), (2, 15)]


def test_nothing_is_removed_and_unknown_settings_are_ignored():
    c = Curriculum()
    fill(c, (1, 10), 200)
    c.advance()
    fill(c, (2, 10), 0)
    c.record([4], [40], [True])
    c.advance()
    assert c.levels == [(1, 10), (2, 10), (1, 15)]
    assert (4, 40) not in c.stat_dict


def test_constructor_arguments():
    c = Curriculum(init_set=(2, 20), window=10, pass_rate=0.5, agent_step=2, map_step=10, max_num_agents=6, max_map_length=40)
    fill(c, (2, 20), 5, 10)
    assert c.advance() == [(4, 20), (2, 30)]


def _padded(n, N, rng, torch):
    """obs / comm of an n-agent batch and the same padded to N agents (absent rows and columns zero)."""
    B = 3
    obs = torch.as_tensor(rng.integers(0, 2, size=(B, n, 6, 9, 9)).astype(np.uint8))
    comm = torch.as_tensor(rng.integers(0, 2, size=(B, n, n)).astype(np.uint8))
    comm |= torch.eye(n, dtype=torch.uint8)[None]
    obs_p = torch.zeros((B, N, 6, 9, 9), dtype=torch.uint8)
    obs_p[:, :n] = obs
    comm_p = torch.zeros((B, N, N), dtype=torch.uint8)
    comm_p[:, :n, :n] = comm
    return obs, comm, obs_p, comm_p


@pytest.mark.parametrize("n", [1, 3, 5])
def test_qnet_step_and_bootstrap_ignore_absent_agents(n):
    torch = pytest.importorskip("torch")
    from mapf_rl_b200.qnet import Network
    torch.manual_seed(0)
    net = Network().eval()
    rng = np.random.default_rng(n)
    N = 6
    # step, twice (the recurrent state carries over)
    a = Network().eval()
    a.load_state_dict(net.state_dict())
    for _ in range(2):
        obs, comm, obs_p, comm_p = _padded(n, N, rng, torch)
        act, q, hid = net.step(obs, comm)
        act_p, q_p, hid_p = a.step(obs_p, comm_p)
        np.testing.assert_allclose(q_p[:, :n].numpy(), q.numpy(), rtol=1e-5, atol=1e-5)
        np.testing.assert_allclose(hid_p[:, :n].numpy(), hid.numpy(), rtol=1e-5, atol=1e-5)
    # bootstrap over T frames
    B, T = 3, 4
    obs = torch.as_tensor(rng.integers(0, 2, size=(B, T, n, 6, 9, 9)).astype(np.uint8))
    comm = torch.as_tensor(rng.integers(0, 2, size=(B, T, n, n)).astype(np.uint8)) | torch.eye(n, dtype=torch.uint8)
    hidden = torch.randn(B, n, 256)
    obs_p = torch.zeros((B, T, N, 6, 9, 9), dtype=torch.uint8)
    obs_p[:, :, :n] = obs
    comm_p = torch.zeros((B, T, N, N), dtype=torch.uint8)
    comm_p[:, :, :n, :n] = comm
    hidden_p = hidden[:, :1].expand(B, N, 256).clone()       # the store broadcasts agent 0's vector to every row
    hidden_p[:, :n] = hidden
    steps = torch.tensor([1, 3, 4])
    with torch.no_grad():
        q = net.bootstrap(obs, steps, hidden.reshape(B * n, 256), comm)
        q_p = net.bootstrap(obs_p, steps, hidden_p.reshape(B * N, 256), comm_p)
    np.testing.assert_allclose(q_p.numpy(), q.numpy(), rtol=1e-5, atol=1e-5)
