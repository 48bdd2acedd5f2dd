"""Packed observations and communication masks of the compact replay store (include/mapf_b200.h, DESIGN.md §3).

- Observation: one 64-byte row per agent.  Element k = c*81 + r*9 + col of the agent's flattened 6x9x9 bool observation is
  bit k & 7 of byte k >> 3, LSB first: np.packbits(obs.reshape(N, 486), axis=-1, bitorder="little") padded to 64 bytes.
  Bits 486..511 are always 0.
- Comm mask: agent i's row is ceil(N/8) bytes, bit j (LSB first) = mask[i][j].

`unpack_obs` is the device kernel (mapf_obs_unpack); the numpy functions restate the formats for `ReplayStore.add` and tests.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _native, config

OBS_ELEMS = int(np.prod(config.obs_shape))   # 486
OBS_BYTES = 64                               # MAPF_OBS_PACKED_BYTES_PER_AGENT


def comm_bytes(num_agents: int) -> int:
    """Bytes of one agent's packed comm-mask row."""
    return (int(num_agents) + 7) // 8


def pack_obs(obs) -> np.ndarray:
    """bool observations [..., N, 6, 9, 9] -> packed rows uint8 [..., N, 64]."""
    obs = np.asarray(obs)
    flat = (obs.reshape(*obs.shape[:-3], OBS_ELEMS) != 0)
    bits = np.packbits(flat, axis=-1, bitorder="little")                   # 61 bytes, the last 2 bits 0
    out = np.zeros((*bits.shape[:-1], OBS_BYTES), dtype=np.uint8)
    out[..., :bits.shape[-1]] = bits
    return out


def unpack_obs_np(bits) -> np.ndarray:
    """packed rows uint8 [..., N, 64] -> uint8 0 / 1 observations [..., N, 6, 9, 9] (pad bits ignored)."""
    bits = np.asarray(bits, dtype=np.uint8)
    flat = np.unpackbits(bits, axis=-1, bitorder="little")[..., :OBS_ELEMS]
    return flat.reshape(*bits.shape[:-1], *config.obs_shape)


def pack_comm(mask) -> np.ndarray:
    """comm masks [..., N, N] -> packed rows uint8 [..., N, ceil(N/8)]."""
    return np.packbits(np.asarray(mask) != 0, axis=-1, bitorder="little")


def unpack_comm(bits, num_agents: int) -> np.ndarray:
    """packed rows uint8 [..., N, ceil(N/8)] -> uint8 0 / 1 masks [..., N, num_agents]."""
    return np.unpackbits(np.asarray(bits, dtype=np.uint8), axis=-1, bitorder="little")[..., :int(num_agents)]


def single_hidden(hid) -> np.ndarray:
    """Hidden rows [T, N, latent] of T transitions -> their one vector each [T, latent].  Raises ValueError if the rows of a
    transition differ: the reference writes agent 0's vector into every row (buffer.py:148), and a compact store keeps one."""
    hid = np.asarray(hid)
    if hid.size and not (hid == hid[:, :1]).all():
        raise ValueError("a compact store keeps one hidden vector per transition, but the hidden rows of one transition differ")
    return hid[:, 0]


_DTYPES = None


def unpack_obs(bits, rows=None, dtype=None):
    """Packed frames -> dense observations on the device (mapf_obs_unpack, one launch).
    bits: uint8 CUDA tensor [F, N, 64] (e.g. `ReplayStore.obs_bits`); rows: int64 CUDA tensor [count] of frames to read
    (default: all F, in order).  Returns [count, N, 6, 9, 9] of `dtype` (torch.uint8 (default), float16 or bfloat16)."""
    import torch
    global _DTYPES
    if _DTYPES is None:
        _DTYPES = {torch.uint8: _native.DTYPE_U8, torch.float16: _native.DTYPE_F16, torch.bfloat16: _native.DTYPE_BF16}
    dtype = torch.uint8 if dtype is None else dtype
    if dtype not in _DTYPES:
        raise ValueError(f"unpack_obs: dtype must be uint8, float16 or bfloat16, got {dtype}")
    assert bits.is_cuda and bits.dtype == torch.uint8 and bits.is_contiguous() and bits.dim() == 3 and bits.shape[2] == OBS_BYTES
    N = int(bits.shape[1])
    rows_ptr = None
    count = int(bits.shape[0])
    if rows is not None:
        assert rows.dtype == torch.int64 and rows.is_cuda and rows.is_contiguous() and rows.dim() == 1
        rows_ptr = C.c_void_p(rows.data_ptr())
        count = int(rows.numel())
    out = torch.empty((count, N, *config.obs_shape), dtype=dtype, device=bits.device)
    lib = _native.lib()
    stream = C.c_void_p(torch.cuda.current_stream(bits.device).cuda_stream)
    _native.check(lib.mapf_obs_unpack(C.c_void_p(bits.data_ptr()), rows_ptr, count, N, _DTYPES[dtype],
                                      C.c_void_p(out.data_ptr()), stream))
    return out
