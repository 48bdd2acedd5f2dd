"""Plain numpy restatement of the device instance generator, `reset_env_warp` (mapf_rl_b200/csrc/mapf_reset_device.cuh).

The device generator is counter-based: instance g of seed s is a pure function of (s, g, L, N, density), so it can be
restated on the host bit for bit and every generated environment compared with it, not just its distribution.  The rules
as the kernel implements them:

* Philox4x32-10 with key (seed & 0xffffffff, seed >> 32); counter (g_lo, g_hi, purpose | attempt << 8, index).
* density None: u = (x >> 8) * 2^-24 from counter (g, 0, 0), inverse CDF of triangular(0, 0.33, 0.5) in float32; the
  obstacle threshold is trunc(density * 2^32) with 0 and 0xffffffff at the ends.
* map: one Philox call per row and per 4 columns (purpose 1, index row * 64 + col / 4); cell col + j is free iff output
  word j >= threshold.
* eligible cells: free cells with a free 4-neighbour; components are the 4-connected components of the free cells.
* agent i (purpose 2, index i): r.x picks the start, r.y the goal, each as the r-th set cell with r = (rnd * total) >> 32
  in LANE-MAJOR order (row % 32, row // 32, col): the warp holds row `lane + 32 q` in lane `lane`.
* the start leaves the eligible set; the goal is picked among the eligible cells of the start's component and leaves
  it too; a component left with fewer than 2 eligible cells is dropped.
* no eligible start cell: the whole instance is redrawn with attempt + 1; 256 failed attempts are an error.
"""
import numpy as np
from scipy import ndimage

M32 = 0xFFFFFFFF
PURPOSE_DENSITY, PURPOSE_MAP, PURPOSE_AGENT = 0, 1, 2
MAX_ATTEMPTS = 256


class GeneratorFailed(RuntimeError):
    pass


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 of counter words c0..c3 (scalars or arrays) under key (k0, k1) -> four uint64 arrays of 32-bit words."""
    c0, c1, c2, c3 = (np.asarray(c, dtype=np.uint64) & M32 for c in (c0, c1, c2, c3))
    c0, c1, c2, c3 = np.broadcast_arrays(c0, c1, c2, c3)
    k0, k1 = int(k0) & M32, int(k1) & M32
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c0
        p1 = np.uint64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ np.uint64(k0), p1 & np.uint64(M32), \
            (p0 >> np.uint64(32)) ^ c3 ^ np.uint64(k1), p0 & np.uint64(M32)
        k0 = (k0 + 0x9E3779B9) & M32
        k1 = (k1 + 0xBB67AE85) & M32
    return c0, c1, c2, c3


def instance_density(seed, g, density):
    """float32 density of instance g: `density` as the library receives it (a C float), or the triangular draw."""
    if density is not None and density >= 0:
        return np.float32(density)
    x = int(philox4x32_10(g & M32, g >> 32, PURPOSE_DENSITY, 0, seed & M32, seed >> 32)[0])
    f = np.float32
    u = f(x >> 8) * f(1.0 / 16777216.0)
    if u < f(0.66):
        return np.sqrt(u * f(0.5) * f(0.33))
    return f(0.5) - np.sqrt((f(1.0) - u) * f(0.5) * f(0.17))


def threshold(dens):
    dens = np.float32(dens)
    if dens <= 0:
        return 0
    if dens >= 1:
        return M32
    return int(float(dens) * 4294967296.0)


def pick_order(L):
    """Rows in the order the warp's pick visits them: lane-major (row % 32, row // 32)."""
    return np.array(sorted(range(L), key=lambda r: (r % 32, r // 32)), dtype=np.int64)


def draw_map(seed, g, L, thresh, attempt):
    """-> bool[L, L], True = free."""
    W = (L + 3) // 4
    rows = np.arange(L, dtype=np.uint64)[:, None]
    quads = np.arange(W, dtype=np.uint64)[None, :]
    words = philox4x32_10(g & M32, g >> 32, PURPOSE_MAP | (attempt << 8), rows * np.uint64(64) + quads, seed & M32, seed >> 32)
    free = np.stack(words, axis=-1) >= np.uint64(thresh)      # [L, W, 4]: cell 4 q + j
    return free.reshape(L, 4 * W)[:, :L]


def generate(seed, g, L, N, density, order=None):
    """Instance g of `seed` as reset_env_warp draws it.  density None = triangular draw.
    -> (map uint8[L,L] (1 = obstacle), starts uint8[N,2], goals uint8[N,2], attempts before the one that succeeded).
    `order`: rows in pick order (default: lane-major, `pick_order(L)`)."""
    seed, g = int(seed), int(g)
    thresh = threshold(instance_density(seed, g, density))
    rows = pick_order(L) if order is None else order
    for attempt in range(MAX_ATTEMPTS):
        free = draw_map(seed, g, L, thresh, attempt)
        nb = np.zeros_like(free)
        nb[1:] |= free[:-1]
        nb[:-1] |= free[1:]
        nb[:, 1:] |= free[:, :-1]
        nb[:, :-1] |= free[:, 1:]
        label, _ = ndimage.label(free)                          # 4-connected (the default cross structure)
        # everything below works on cells ranked in pick order: k -> (rows[k // L], k % L)
        elig = (free & nb)[rows].ravel()
        comp = label[rows].ravel()
        draws = philox4x32_10(g & M32, g >> 32, PURPOSE_AGENT | (attempt << 8), np.arange(N, dtype=np.uint64),
                              seed & M32, seed >> 32)
        rx, ry = (d.astype(np.int64) for d in draws[:2])
        starts = np.zeros((N, 2), dtype=np.uint8)
        goals = np.zeros((N, 2), dtype=np.uint8)
        ok = True
        for i in range(N):
            cells = np.flatnonzero(elig)
            if len(cells) == 0:
                ok = False
                break
            s = cells[(int(rx[i]) * len(cells)) >> 32]
            elig[s] = False
            in_comp = comp == comp[s]
            cand = np.flatnonzero(elig & in_comp)               # never empty: a component keeps >= 2 eligible cells
            t = cand[(int(ry[i]) * len(cand)) >> 32]
            elig[t] = False
            if len(cand) - 1 < 2:
                elig[in_comp] = False
            starts[i] = rows[s // L], s % L
            goals[i] = rows[t // L], t % L
        if ok:
            return (~free).astype(np.uint8), starts, goals, attempt
    raise GeneratorFailed(f"no instance after {MAX_ATTEMPTS} attempts (seed {seed}, g {g}, L {L}, N {N}, density {density})")


def generate_batch(seed, env_offset, B, L, N, density):
    """Slots 0..B-1 of reset(seed, env_offset): instance env_offset + e each.  -> (maps, starts, goals, attempts[B])."""
    out = [generate(seed, env_offset + e, L, N, density) for e in range(B)]
    return (np.stack([o[0] for o in out]), np.stack([o[1] for o in out]), np.stack([o[2] for o in out]),
            np.array([o[3] for o in out]))
