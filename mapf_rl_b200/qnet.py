"""Batched restatement of the reference Q-network's inference glue (model.py:139-263) in plain PyTorch.

The network itself is OUT OF SCOPE of the hand-written kernels (its GEMMs / convolutions stay in PyTorch,
BASELINE.json north star); this module exists because the reference `Network.step` handles ONE environment per
call (model.py:181-222, batch dim 1) and `CommBlock` hard-codes `config.batch_size` (model.py:128), which would
make a batched actor host-bound.  Sub-module names, shapes and construction order are those of the
reference, so a reference checkpoint (`torch.save(model.state_dict())`, worker.py:338) loads unchanged and a
same-seed initialisation draws the same weights.  The communication mask comes from the CUDA kernel
(`BatchedEnvironment.comm_mask`) instead of the per-env topk of model.py:196-208.

For throughput run it as `Network().cuda().eval().to(memory_format=torch.channels_last)` under
`torch.autocast("cuda", torch.bfloat16)`: 2048 envs x 32 agents take 38 ms in fp32, 24.6 ms with bf16 autocast and
15.7 ms with NHWC weights on a B200 (profiles/qnet_forward_probe.py) -- still ~700x the env step it follows.
"""
from __future__ import annotations

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import config

NUM_COMM_LAYERS = 2   # config.py:61
NUM_COMM_HEADS = 2    # config.py:62


class ResBlock(nn.Module):  # model.py:7-42, type='cnn', bn=False (the only variant the reference instantiates)
    def __init__(self, channel):
        super().__init__()
        self.block1 = nn.Conv2d(channel, channel, 3, 1, 1)
        self.block2 = nn.Conv2d(channel, channel, 3, 1, 1)

    def forward(self, x):
        return F.relu(self.block2(F.relu(self.block1(x))) + x)


class MultiHeadAttention(nn.Module):  # model.py:45-86
    def __init__(self, input_dim, output_dim, num_heads):
        super().__init__()
        self.num_heads, self.input_dim, self.output_dim = num_heads, input_dim, output_dim
        self.W_Q = nn.Linear(input_dim, output_dim * num_heads)
        self.W_K = nn.Linear(input_dim, output_dim * num_heads)
        self.W_V = nn.Linear(input_dim, output_dim * num_heads)
        self.W_O = nn.Linear(output_dim * num_heads, output_dim, bias=False)

    def forward(self, x, attn_mask):
        B, N, _ = x.shape
        q = self.W_Q(x).view(B, N, self.num_heads, -1).transpose(1, 2)
        k = self.W_K(x).view(B, N, self.num_heads, -1).transpose(1, 2)
        v = self.W_V(x).view(B, N, self.num_heads, -1).transpose(1, 2)
        # scores in fp32 whatever the autocast state (model.py:75-78)
        scores = torch.matmul(q.float(), k.float().transpose(-1, -2)) / (self.output_dim ** 0.5)
        scores = scores.masked_fill(attn_mask.unsqueeze(1), -1e9)
        attn = F.softmax(scores, dim=-1)
        ctx = torch.matmul(attn.to(v.dtype), v).transpose(1, 2).contiguous().view(B, N, self.num_heads * self.output_dim)
        return self.W_O(ctx)


class CommBlock(nn.Module):  # model.py:88-135, for any batch size
    def __init__(self, input_dim, output_dim=64, num_heads=NUM_COMM_HEADS, num_layers=NUM_COMM_LAYERS):
        super().__init__()
        self.input_dim, self.output_dim, self.num_layers = input_dim, output_dim, num_layers
        self.self_attn = MultiHeadAttention(input_dim, output_dim, num_heads)
        self.update_cell = nn.GRUCell(output_dim, input_dim)

    def forward(self, latent, comm_mask):
        """latent [B,N,D]; comm_mask bool [B,N,N].  Agents with more than one partner (themselves included) are
        updated (model.py:97-99, 123-133); the others keep their latent — without the data-dependent early exit
        of model.py:101-103 (identical result, no host sync)."""
        B, N, D = latent.shape
        update_mask = (comm_mask.sum(dim=-1) > 1).unsqueeze(2)
        attn_mask = ~comm_mask
        for _ in range(self.num_layers):
            info = self.self_attn(latent, attn_mask)
            upd = self.update_cell(info.reshape(-1, self.output_dim).to(latent.dtype), latent.reshape(-1, D)).view(B, N, D)
            latent = torch.where(update_mask, upd, latent)
        return latent


class Network(nn.Module):
    """model.Network (model.py:139-263) with batched `step` / `bootstrap`."""

    def __init__(self):
        super().__init__()
        self.latent_dim = config.latent_dim
        self.obs_encoder = nn.Sequential(
            nn.Conv2d(config.obs_shape[0], 128, 3, 1), nn.ReLU(True),
            ResBlock(128), ResBlock(128), ResBlock(128),
            nn.Conv2d(128, 16, 1, 1), nn.ReLU(True), nn.Flatten())
        self.recurrent = nn.GRUCell(16 * 7 * 7, self.latent_dim)
        self.comm = CommBlock(self.latent_dim)
        self.adv = nn.Linear(self.latent_dim, 5)
        self.state = nn.Linear(self.latent_dim, 1)
        self.hidden = None
        for _, m in self.named_modules():  # model.py:175-179
            if isinstance(m, (nn.Linear, nn.Conv2d)):
                nn.init.xavier_uniform_(m.weight)
                if m.bias is not None:
                    nn.init.constant_(m.bias, 0)

    def _q(self, hidden):
        adv = self.adv(hidden)
        return self.state(hidden) + adv - adv.mean(-1, keepdim=True)   # model.py:216-219

    @torch.no_grad()
    def step(self, obs, comm_mask, reset_mask=None, present=None):
        """obs uint8/float [B,N,6,9,9], comm_mask uint8/bool [B,N,N] (BatchedEnvironment.comm_mask),
        reset_mask bool [B] (optional): environments whose recurrent state restarts (Network.reset, model.py:224).
        -> (actions int64[B,N], q [B,N,5], hidden [B,N,256]); the recurrent state is kept in self.hidden.
        present (`present.PresentRows`): obs is [M_pad,6,9,9] in present rows; the encoder and the input GRU run on those rows
        only, the comm block and the head on the padded [B,N] layout, and absent agents' hidden state, q and actions are 0."""
        B, N = comm_mask.shape[:2]
        p = next(self.parameters())
        x = obs if present is not None else obs.reshape(B * N, *obs.shape[2:])
        latent = self.obs_encoder(x.to(p.dtype))
        if self.hidden is None or self.hidden.shape[0] != B * N:
            self.hidden = torch.zeros(B * N, self.latent_dim, dtype=p.dtype, device=p.device)   # GRUCell(x) == GRUCell(x, 0)
        elif reset_mask is not None:
            keep = (~reset_mask.bool()).to(p.dtype).repeat_interleave(N).unsqueeze(1)
            self.hidden = self.hidden * keep
        if present is None:
            hidden = self.recurrent(latent, self.hidden).view(B, N, self.latent_dim)
        else:
            h = self.recurrent(latent[:present.M], present.gather(self.hidden))
            hidden = present.scatter(h).view(B, N, self.latent_dim)
        hidden = self.comm(hidden, comm_mask.bool())
        self.hidden = hidden.reshape(B * N, self.latent_dim)
        q = self._q(hidden)
        if present is not None:
            q = torch.where(present.mask.unsqueeze(-1), q, torch.zeros_like(q))
        return q.argmax(-1), q, hidden

    def reset(self):
        self.hidden = None

    def bootstrap(self, obs, steps, hidden, comm_mask, present=None):
        """model.py:227-263 for any batch size: obs [B,T,N,6,9,9], steps int64[B] (1-based frame whose hidden is
        read out), hidden [B*N,256], comm_mask bool [B,T,N,N] -> q of agent 0, [B,5].
        present (`present.PresentRows`): obs [M_pad,T,6,9,9] and hidden [M_pad,256] in present rows
        (`ReplayStore.gather(idx, present=True)`); the encoder and the input GRU run on those rows, the comm block on the
        padded layout of each frame."""
        B, T, N = comm_mask.shape[:3]
        p = next(self.parameters())
        if present is None:
            x = obs.transpose(1, 2).contiguous().view(-1, *obs.shape[3:]).to(p.dtype)
            latent = self.obs_encoder(x).view(B * N, T, 16 * 7 * 7).transpose(0, 1)
            hidden = hidden.to(p.dtype)
        else:
            latent = self.obs_encoder(obs.reshape(-1, *obs.shape[2:]).to(p.dtype)).view(-1, T, 16 * 7 * 7)
            latent = latent[:present.M].transpose(0, 1)
            hidden = hidden[:present.M].to(p.dtype)
        buf = []
        for i in range(T):
            hidden = self.recurrent(latent[i].to(hidden.dtype), hidden)
            if present is not None:
                hidden = present.scatter(hidden)
            hidden = self.comm(hidden.view(B, N, self.latent_dim), comm_mask[:, i].bool())
            buf.append(hidden[:, 0])
            hidden = hidden.reshape(B * N, self.latent_dim)
            if present is not None:
                hidden = present.gather(hidden)
        buf = torch.stack(buf).transpose(0, 1)
        h = buf[torch.arange(B, device=buf.device), steps - 1]
        return self._q(h)
