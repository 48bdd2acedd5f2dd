"""The batched PyTorch restatement of the Q-network glue (mapf_rl_b200/qnet.py) against the live reference
model (model.py:139-263), CPU fp32, where the reference is installed (MAPF_REFERENCE_DIR); the architecture test runs
everywhere.  The network is outside the hand-written kernels; this pins that a reference checkpoint / seed gives the
same Q-values through the batched path, to fp32 round-off (1e-5 relative)."""
import numpy as np
import pytest
import torch

from helpers import instances
from oracle import oracle, ref_loader

needs_reference = pytest.mark.skipif(not ref_loader.available(), reason="the reference is not installed (MAPF_REFERENCE_DIR)")


def nets():
    from mapf_rl_b200 import qnet
    model = ref_loader.load_module("model")
    torch.manual_seed(3)
    ref = model.Network().eval()
    torch.manual_seed(3)
    mine = qnet.Network().eval()
    return ref, mine


def test_architecture_of_reference_model():
    """Without the reference: the layer shapes and the parameter count SURVEY.md section 2 took from model.py:147-170
    (conv 6->128 3x3, three residual blocks, 1x1 conv ->16, GRUCell 784->256, 2-head attention comm block with a GRU
    update, dueling head over 5 actions; 2,050,582 parameters), so a reference checkpoint still has a place for every tensor."""
    from mapf_rl_b200 import qnet
    sd = qnet.Network().state_dict()
    assert tuple(sd["obs_encoder.0.weight"].shape) == (128, 6, 3, 3)
    assert [tuple(sd[f"obs_encoder.{i}.block{j}.weight"].shape) for i in (2, 3, 4) for j in (1, 2)] == [(128, 128, 3, 3)] * 6
    assert tuple(sd["obs_encoder.5.weight"].shape) == (16, 128, 1, 1)
    assert tuple(sd["recurrent.weight_ih"].shape) == (3 * 256, 16 * 7 * 7) and tuple(sd["recurrent.weight_hh"].shape) == (3 * 256, 256)
    assert tuple(sd["comm.update_cell.weight_hh"].shape) == (3 * 256, 256)
    assert tuple(sd["adv.weight"].shape) == (5, 256) and tuple(sd["state.weight"].shape) == (1, 256)
    assert sum(v.numel() for v in sd.values()) == 2050582


@needs_reference
def test_same_seed_same_weights_and_checkpoint_compatible():
    ref, mine = nets()
    sd_r, sd_m = ref.state_dict(), mine.state_dict()
    assert list(sd_r.keys()) == list(sd_m.keys())
    for k in sd_r:
        assert torch.equal(sd_r[k], sd_m[k]), k
    mine.load_state_dict(sd_r)  # a reference checkpoint loads unchanged (worker.py:338)
    assert sum(p.numel() for p in mine.parameters()) == 2050582  # SURVEY section 2


@needs_reference
def test_step_matches_reference_per_env():
    ref, mine = nets()
    maps, agents, goals = instances(16)
    envs = []
    for k in (0, 9, 33):
        o = oracle.OracleEnv()
        o.load(maps[k], agents[k], goals[k])
        envs.append(o)
    refs = []
    for _ in envs:   # one reference network per environment (worker.py:359-361)
        torch.manual_seed(3)
        r = ref_loader.load_module("model").Network().eval()
        r.load_state_dict(ref.state_dict())
        refs.append(r)
    rng = np.random.default_rng(0)
    mine.reset()
    for s in range(4):
        obs = np.stack([e.observe()[0] for e in envs]).astype(np.float32)
        pos = np.stack([e.observe()[1] for e in envs]).astype(np.float32)
        outs = [refs[i].step(torch.from_numpy(obs[i]), torch.from_numpy(pos[i])) for i in range(len(envs))]
        comm = np.stack([o[3] for o in outs])                       # the reference's own mask (ties as torch.topk broke them)
        act, q, hid = mine.step(torch.from_numpy(obs), torch.from_numpy(comm))
        for i, (a_ref, q_ref, h_ref, _) in enumerate(outs):
            np.testing.assert_allclose(q[i].numpy(), q_ref, rtol=1e-5, atol=1e-5)
            np.testing.assert_allclose(hid[i].numpy(), h_ref, rtol=1e-5, atol=1e-5)
        for i, e in enumerate(envs):
            e.step(rng.integers(0, 5, size=16))


@needs_reference
def test_bootstrap_matches_reference():
    ref, mine = nets()
    cfg = ref_loader.load_module("config")
    B, T, N = cfg.batch_size, 3, 2          # the reference hard-codes config.batch_size (model.py:241,128)
    g = torch.Generator().manual_seed(1)
    obs = (torch.rand(B, T, N, 6, 9, 9, generator=g) < 0.2).float()
    comm = torch.rand(B, T, N, N, generator=g) < 0.5
    comm = comm | torch.eye(N, dtype=torch.bool)
    hidden = torch.randn(B * N, 256, generator=g) * 0.1
    steps = torch.randint(1, T + 1, (B,), generator=g)
    with torch.no_grad():
        q_ref = ref.bootstrap(obs.clone(), steps, hidden.clone(), comm.clone())
        q_mine = mine.bootstrap(obs, steps, hidden, comm)
    np.testing.assert_allclose(q_mine.numpy(), q_ref.float().numpy(), rtol=1e-5, atol=1e-5)
