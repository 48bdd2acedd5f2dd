"""CPU: the present-row format (mapf_rl_b200/present.py) against its numpy restatement, and Network.step / bootstrap on present
rows against the padded network (fp32, within 1e-5)."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from mapf_rl_b200 import present  # noqa: E402
from mapf_rl_b200.present import PresentRows, present_np  # noqa: E402

N = 6
COUNTS = {
    "all1": [1] * 7,
    "allN": [N] * 5,
    "random": list(np.random.default_rng(3).integers(1, N + 1, size=11)),
    "alternating": [1, N] * 4,
}


@pytest.mark.parametrize("name", list(COUNTS))
def test_rows_offsets_and_padding_match_numpy(name):
    counts = np.asarray(COUNTS[name], dtype=np.int64)
    pr = PresentRows(torch.as_tensor(counts.astype(np.uint8)), int(counts.sum()), N)
    first, index, M, M_pad = present_np(counts, N)
    assert pr.M == M == int(counts.sum()) and pr.M_pad == M_pad and pr.B == len(counts)
    assert M_pad % present.QUANTUM == 0 and M <= M_pad < M + present.QUANTUM
    assert np.array_equal(pr.first.numpy(), first) and pr.first.dtype == torch.int32
    assert np.array_equal(pr.index.numpy(), index)
    # the restatement itself: row first[e] + a is agent a of environment e
    for e, n in enumerate(counts):
        for a in range(n):
            assert index[first[e] + a] == e * N + a
    assert np.array_equal(pr.mask.numpy(), np.arange(N)[None, :] < counts[:, None])
    # select / scatter / gather
    x = torch.randn(len(counts) * N, 3)
    sel = pr.select(x)
    assert sel.shape == (M_pad, 3)
    assert torch.equal(sel[:M], x[torch.as_tensor(index)]) and not sel[M:].any()
    back = pr.scatter(sel[:M])
    assert torch.equal(back.view(len(counts), N, 3)[pr.mask], x.view(len(counts), N, 3)[pr.mask])
    assert not back.view(len(counts), N, 3)[~pr.mask].any()
    assert torch.equal(pr.gather(back), sel[:M])


def _net_pair():
    from mapf_rl_b200.qnet import Network
    torch.manual_seed(0)
    a = Network().eval()
    with torch.no_grad():   # non-zero head biases: absent agents' q is 0 only because the present path zeroes it
        a.adv.bias.uniform_(-1, 1)
        a.state.bias.uniform_(-1, 1)
    b = Network().eval()
    b.load_state_dict(a.state_dict())
    return a, b


def _frames(rng, counts, shape_tail=(6, 9, 9)):
    B = len(counts)
    obs = torch.as_tensor(rng.integers(0, 2, size=(B, N, *shape_tail)).astype(np.uint8))
    comm = torch.as_tensor(rng.integers(0, 2, size=(B, N, N)).astype(np.uint8)) | torch.eye(N, dtype=torch.uint8)
    m = torch.as_tensor(np.arange(N)[None, :] < np.asarray(counts)[:, None])
    obs = obs * m[:, :, None, None, None]
    comm = comm * (m[:, :, None] & m[:, None, :])
    return obs, comm


def _step_twin(quantum, monkeypatch):
    monkeypatch.setattr(present, "QUANTUM", quantum)
    padded, pres = _net_pair()
    rng = np.random.default_rng(11)
    counts = np.asarray([6, 1, 3, 6, 2, 5], dtype=np.int64)
    outs = []
    for s in range(3):
        reset = None
        if s == 2:   # environments 0 and 3 restart with fewer agents, environment 1 with more
            reset = torch.tensor([True, True, False, True, False, False])
            counts = counts.copy()
            counts[[0, 1, 3]] = [2, 4, 1]
        obs, comm = _frames(rng, counts)
        pr = PresentRows(torch.as_tensor(counts), int(counts.sum()), N)
        ap, qp, hp = padded.step(obs, comm, reset_mask=reset)
        x = pr.select(obs.flatten(0, 1))
        a, q, h = pres.step(x, comm, reset_mask=reset, present=pr)
        m = pr.mask
        np.testing.assert_allclose(q[m].numpy(), qp[m].numpy(), rtol=1e-5, atol=1e-5)
        np.testing.assert_allclose(h[m].numpy(), hp[m].numpy(), rtol=1e-5, atol=1e-5)
        # absent agents: exactly 0, also in the recurrent state the next step starts from
        assert not q[~m].any() and not a[~m].any() and not h[~m].any()
        assert not pres.hidden.view(len(counts), N, -1)[~m].any()
        outs.append((q, h))
    return outs


def test_step_present_matches_padded_over_three_steps_with_reset(monkeypatch):
    _step_twin(present.QUANTUM, monkeypatch)


def _bootstrap_case(rng, counts, T):
    B = len(counts)
    obs = torch.as_tensor(rng.integers(0, 2, size=(B, T, N, 6, 9, 9)).astype(np.float32))
    comm = torch.as_tensor(rng.integers(0, 2, size=(B, T, N, N)).astype(np.uint8)) | torch.eye(N, dtype=torch.uint8)
    m = torch.as_tensor(np.arange(N)[None, :] < np.asarray(counts)[:, None])
    obs = obs * m[:, None, :, None, None, None]
    comm = comm * (m[:, None, :, None] & m[:, None, None, :])
    hid = torch.randn(B, 1, 256).expand(B, N, 256) * m[:, :, None]    # the store's one vector per sample
    return obs, comm, hid.reshape(B * N, 256).contiguous()


def _bootstrap_twin(quantum, monkeypatch):
    monkeypatch.setattr(present, "QUANTUM", quantum)
    padded, pres = _net_pair()
    rng = np.random.default_rng(5)
    counts = np.asarray([1, 6, 3, 2, 6, 4, 1], dtype=np.int64)
    T = 5
    obs, comm, hid = _bootstrap_case(rng, counts, T)
    steps = torch.tensor([1, 5, 3, 2, 4, 5, 1])
    pr = PresentRows(torch.as_tensor(counts), int(counts.sum()), N)
    B = len(counts)
    x = pr.select(obs.transpose(1, 2).reshape(B * N, T, 6, 9, 9))
    h = pr.select(hid)
    q_p = padded.bootstrap(obs, steps, hid, comm)
    q = pres.bootstrap(x, steps, h, comm, present=pr)
    np.testing.assert_allclose(q.detach().numpy(), q_p.detach().numpy(), rtol=1e-5, atol=1e-6)
    # gradients of a Huber loss through both
    from mapf_rl_b200.learner import BatchedLearner
    target = torch.randn(B, 5)
    grads = []
    for net, qq in ((padded, q_p), (pres, q)):
        net.zero_grad()
        BatchedLearner.huber(qq - target).mean().backward()
        grads.append({k: p.grad.clone() for k, p in net.named_parameters() if p.grad is not None})
    assert grads[0].keys() == grads[1].keys() and len(grads[0]) > 10
    for k in grads[0]:
        g0, g1 = grads[0][k], grads[1][k]
        scale = g0.abs().max().clamp_min(1e-12)
        assert ((g1 - g0).abs().max() / scale) < 1e-5, k
    return q


def test_bootstrap_present_matches_padded_with_gradients(monkeypatch):
    _bootstrap_twin(present.QUANTUM, monkeypatch)


@pytest.mark.parametrize("quantum", [1, 8, 64])
def test_quantum_changes_nothing(quantum, monkeypatch):
    base_step = _step_twin(present.QUANTUM, monkeypatch)
    base_boot = _bootstrap_twin(present.QUANTUM, monkeypatch)
    other_step = _step_twin(quantum, monkeypatch)
    other_boot = _bootstrap_twin(quantum, monkeypatch)
    for (q0, h0), (q1, h1) in zip(base_step, other_step):
        np.testing.assert_allclose(q1.numpy(), q0.numpy(), rtol=1e-5, atol=1e-6)
        np.testing.assert_allclose(h1.numpy(), h0.numpy(), rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(other_boot.detach().numpy(), base_boot.detach().numpy(), rtol=1e-5, atol=1e-6)
    pr = PresentRows(torch.tensor([3, 1, 6]), 10, N)
    assert pr.M_pad == -(-10 // quantum) * quantum
