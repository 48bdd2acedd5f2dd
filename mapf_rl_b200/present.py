"""Present-agent rows: the batch layout in which the Q-network's encoder and input GRU see only the agents that exist.

On a sized environment batch (`BatchedEnvironment(..., sized=True)`) environment e has n_e <= N agents, and its absent agents'
rows are zeros that the padded network encodes and throws away.  In the present layout, environment (or sample) e's agent
a < n_e is row `first[e] + a` of a `[M_pad, ...]` tensor, with `first` the exclusive prefix sum of the counts and M = sum n_e.
Rows M..M_pad-1 are zeros: M_pad rounds M up to QUANTUM because every distinct batch size is a new convolution shape with its
own cuDNN execution plan, and a training run would otherwise meet thousands of them.  Padding rows are encoded and dropped,
never scattered.

`PresentRows` holds the mapping on the device; `unpack_obs_present` is the device kernel that writes a batch of current frames
in this layout (mapf_obs_unpack_present), and `ReplayStore.gather(idx, present=True)` the learner's windows
(mapf_replay_gather_present).  `present_np` restates the format with numpy for the tests.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _native, config

# rows M_pad is a multiple of.  Measured on a B200 (DESIGN.md §4, present-agent batches): the bf16 encoder's first call at a
# new batch size takes 8-264 ms, a steady call about 0.6 us per row.  256 rows of padding cost at most ~0.15 ms a step (under
# 3 % of the encoder at 8192 x 6) and bound the distinct shapes of a run to B * N / 256 (192 at 8192 x 6).
QUANTUM = 256


def padded_rows(M: int) -> int:
    """M rounded up to a multiple of QUANTUM (0 stays 0)."""
    return -(-int(M) // QUANTUM) * QUANTUM


class PresentRows:
    """The present rows of a batch of B environments (or samples) of at most N agents each.

    counts  int64 [B]   agents of each environment, 1..N
    first   int32 [B]   its first row (exclusive prefix sum of counts)
    index   int64 [M]   flat padded index e * N + a of each present row, in row order
    mask    bool [B, N] a < counts[e]
    M, M_pad            host ints
    """

    def __init__(self, counts, M: int, N: int):
        """counts: integer CUDA (or CPU) tensor [B]; M: its sum, read on the host by the caller (the one place a host value is
        needed: it sizes the output tensors)."""
        import torch
        self.N, self.M, self.M_pad = int(N), int(M), padded_rows(M)
        self.counts = counts.to(torch.int64)
        self.B = int(self.counts.numel())
        dev = self.counts.device
        end = torch.cumsum(self.counts, 0)
        self.first = (end - self.counts).to(torch.int32)
        e = torch.repeat_interleave(torch.arange(self.B, device=dev), self.counts, output_size=self.M)
        a = torch.arange(self.M, device=dev) - self.first.to(torch.int64)[e]
        self.index = e * self.N + a
        self.mask = torch.arange(self.N, device=dev)[None, :] < self.counts[:, None]

    def select(self, padded):
        """Rows of a padded tensor [B * N, ...] -> the present layout [M_pad, ...] (padding rows zeros)."""
        out = padded.new_zeros((self.M_pad, *padded.shape[1:]))
        out[:self.M] = padded.index_select(0, self.index)
        return out

    def scatter(self, rows):
        """Present rows [M, ...] -> the padded layout [B * N, ...] with zeros for absent agents (out of place: autograd
        reaches `rows`)."""
        z = rows.new_zeros((self.B * self.N, *rows.shape[1:]))
        return z.index_copy(0, self.index, rows)

    def gather(self, padded):
        """Padded [B * N, ...] -> present rows [M, ...] (autograd-clean)."""
        return padded.index_select(0, self.index)


def present_np(counts, N: int):
    """numpy restatement: counts [B] -> (first int32 [B], index int64 [M] of e * N + a, M, M_pad)."""
    counts = np.asarray(counts, dtype=np.int64)
    first = np.concatenate([[0], np.cumsum(counts)[:-1]]).astype(np.int32) if counts.size else np.zeros(0, np.int32)
    index = np.asarray([e * int(N) + a for e, n in enumerate(counts) for a in range(n)], dtype=np.int64)
    M = int(counts.sum())
    return first, index, M, padded_rows(M)


_DTYPES = None


def unpack_obs_present(bits, rows, present: PresentRows, dtype=None):
    """Current frames of present agents only, on the device (mapf_obs_unpack_present, one launch).
    bits: uint8 CUDA tensor [F, N, 64] (e.g. `ReplayStore.obs_bits`); rows: int64 CUDA tensor [B] of frames (frame e belongs
    to environment e of `present`).  Returns [M_pad, 6, 9, 9] of `dtype` (torch.uint8 (default), float16 or bfloat16)."""
    import torch
    global _DTYPES
    if _DTYPES is None:
        _DTYPES = {torch.uint8: _native.DTYPE_U8, torch.float16: _native.DTYPE_F16, torch.bfloat16: _native.DTYPE_BF16}
    dtype = torch.uint8 if dtype is None else dtype
    if dtype not in _DTYPES:
        raise ValueError(f"unpack_obs_present: dtype must be uint8, float16 or bfloat16, got {dtype}")
    assert bits.is_cuda and bits.dtype == torch.uint8 and bits.is_contiguous() and bits.dim() == 3 and bits.shape[2] == 64
    assert rows.dtype == torch.int64 and rows.is_cuda and rows.is_contiguous() and rows.numel() == present.B
    N = int(bits.shape[1])
    assert N == present.N, "the frames are laid out for the batch's agent count"
    n8 = present.counts.to(torch.uint8).contiguous()
    first = present.first.contiguous()
    out = torch.empty((present.M_pad, *config.obs_shape), dtype=dtype, device=bits.device)
    stream = C.c_void_p(torch.cuda.current_stream(bits.device).cuda_stream)
    _native.check(_native.lib().mapf_obs_unpack_present(C.c_void_p(bits.data_ptr()), C.c_void_p(rows.data_ptr()),
                                                        C.c_void_p(n8.data_ptr()), C.c_void_p(first.data_ptr()), present.B, N,
                                                        present.M_pad, _DTYPES[dtype], C.c_void_p(out.data_ptr()), stream))
    return out
