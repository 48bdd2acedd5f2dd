"""numpy restatement of the replay store's window gather (GlobalBuffer.sample_batch, worker.py:106-184), one sampled leaf at a
time from the contents of its episode slot.

Working per slot lets a test compare a gather from a store of many GB with no host copy of the store: it keeps the sampled
slots only.  A `Slot` holds what a store keeps for one episode slot g, in the dense layout (worker.py:36-42):

    obs     bool / u8 [S + 1, N, 6, 9, 9]   frames g * (S + 1) + f
    comm    bool / u8 [S + 1, N, N]
    hidden  fp16 [S, N, latent]             rows g * S + t
    action  u8 [S], reward fp16 [S]
    done    bool, size int                  (done_buf[g], size_buf[g])
    agents  int                             the store's agents_buf[g]: present rows of the slot's samples (clamped to N)

A compact store's slot is the same with agents >= n of its episode zeroed and its one hidden vector per transition in every
agent's row.  `tests/test_replay_window_ref.py` ties `gather_ref` to `oracle.OracleReplay`."""
from collections import namedtuple

import numpy as np

from mapf_rl_b200.present import present_np

Geometry = namedtuple("Geometry", "N S bt fwd latent")   # max_num_agents, max_steps, bt_steps, forward_steps, latent_dim
Slot = namedtuple("Slot", "obs comm hidden action reward done size agents")

# window geometries the gathers are tested at: the reference's; every minimum (W = 2); bt = 1 with forward steps past most
# episodes and an odd latent; forward = 1 with N % 8 == 0; W = 64, the present gather's limit; W = 65 (dense and compact only);
# N past 32; odd N with an odd latent; MAPF_MAX_AGENTS agents (16 KB comm-mask frames)
GEOMETRIES = [Geometry(6, 256, 16, 2, 256), Geometry(1, 1, 1, 1, 1), Geometry(3, 8, 1, 3, 7), Geometry(8, 40, 5, 1, 8),
              Geometry(4, 64, 60, 4, 20), Geometry(7, 64, 61, 4, 12), Geometry(33, 32, 16, 2, 256),
              Geometry(127, 16, 4, 3, 9), Geometry(128, 24, 8, 2, 256)]
PRESENT_MAX_W = 64   # bt_steps + forward_steps mapf_replay_gather_present serves


def slot_of(obs, comm, hidden, action, reward, done, size, agents, g, S):
    """Slot g of a store given as arrays in the dense layout (obs [(S+1)*cap, N, 6, 9, 9], hidden [S*cap, N, latent], ...)."""
    f, r = slice(g * (S + 1), (g + 1) * (S + 1)), slice(g * S, (g + 1) * S)
    return Slot(obs[f], comm[f], hidden[r], action[r], reward[r], bool(done[g]), int(size[g]), int(agents[g]))


def edge_steps(size, geo):
    """The steps of an episode of `size` transitions where the window changes shape: its ends, the last steps without
    a full burn-in, the first with one, and the steps whose forward frames reach the episode's end."""
    bt, fwd = geo.bt, geo.fwd
    return sorted(t for t in {0, 1, bt - 2, bt - 1, bt, size - fwd - 1, size - fwd, size - 1} if 0 <= t < size)


def scalars(slot, t, geo):
    """The per-sample scalars of leaf (slot, t): action, reward, done, steps, bt_steps, and `bad` = t >= size."""
    return dict(action=np.int64(slot.action[t]), reward=np.float16(slot.reward[t]),
                done=np.float16(t == slot.size - 1 and slot.done),                                  # :145-148
                steps=np.float16(min(geo.fwd, slot.size - t)), bt_steps=np.int64(min(t + 1, geo.bt)),   # :122, :150
                bad=t >= slot.size)


def window(slot, t, geo):
    """What the gather returns for leaf (slot, t): obs fp16 [W, N, 6, 9, 9], comm_mask u8 [W, N, N], hidden fp16 [N, latent]
    and `scalars`.  The reference asserts t < size (worker.py:120); the device gathers latch such a leaf and still write the
    window of the same formulas, the slot's frames up to `size`."""
    N, W = geo.N, geo.bt + geo.fwd
    steps = min(geo.fwd, slot.size - t)                # :122
    f0 = max(0, t + 1 - geo.bt)                        # :124-137: the window starts at the episode's first frame
    n = max(0, t + 1 + steps - f0)                     #           until bt_steps frames of history exist
    obs = np.zeros((W, N, 6, 9, 9), dtype=np.float16)  # :139-142 zero padding, :169 astype(np.float16)
    comm = np.zeros((W, N, N), dtype=np.uint8)
    obs[:n] = slot.obs[f0:f0 + n]
    comm[:n] = slot.comm[f0:f0 + n]
    if t >= geo.bt:                                    # :137 the hidden state bt_steps before t
        hidden = np.asarray(slot.hidden[t - geo.bt], dtype=np.float16)
    else:                                              # :127, :132
        hidden = np.zeros((N, geo.latent), dtype=np.float16)
    return dict(obs=obs, comm_mask=comm, hidden=hidden, **scalars(slot, t, geo))


SCALARS = ("action", "reward", "done", "steps", "bt_steps", "bad")
BATCHED = ("obs", "comm_mask") + SCALARS


def scalars_ref(slots, idx, geo):
    """`gather_ref`'s scalars alone, for batches whose windows are too large to hold on the host."""
    per = [scalars(slots[leaf // geo.S], leaf % geo.S, geo) for leaf in np.asarray(idx, dtype=np.int64).tolist()]
    return {k: np.asarray([p[k] for p in per]) for k in SCALARS}


def gather_ref(slots, idx, geo):
    """The batch of leaves `idx` (leaf = slot * S + t; `slots` maps a slot id to its `Slot`) as the gathers return it:
    obs [B, W, N, 6, 9, 9], comm_mask [B, W, N, N], hidden [B * N, latent], action / reward / done / steps / bt_steps /
    bad [B], and agents [B], the slot's agents entry of each sample."""
    idx = np.asarray(idx, dtype=np.int64)
    memo = {}
    wins = []
    for leaf in idx.tolist():
        if leaf not in memo:
            memo[leaf] = window(slots[leaf // geo.S], leaf % geo.S, geo)
        wins.append(memo[leaf])
    out = {k: np.stack([w[k] for w in wins]) if wins else np.zeros(0) for k in BATCHED}
    out["hidden"] = np.concatenate([w["hidden"] for w in wins]) if wins else np.zeros((0, geo.latent), np.float16)
    out["agents"] = np.asarray([slots[leaf // geo.S].agents for leaf in idx.tolist()], dtype=np.int64)
    return out


def present_ref(ref, geo, out_rows=None):
    """`gather_ref`'s batch in present-agent rows (mapf_rl_b200/present.py): sample b's agent a < n_b = min(agents_b, N) is row
    first[b] + a of obs [out_rows, W, 6, 9, 9] and hidden [out_rows, latent]; rows past M are zeros.  out_rows defaults to
    M_pad.  -> (obs, hidden, first, M, M_pad)."""
    N, W = geo.N, geo.bt + geo.fwd
    counts = np.minimum(ref["agents"], N)
    first, index, M, M_pad = present_np(counts, N)
    out_rows = M_pad if out_rows is None else int(out_rows)
    B = len(counts)
    obs = np.zeros((out_rows, W, 6, 9, 9), dtype=np.float16)
    hidden = np.zeros((out_rows, geo.latent), dtype=np.float16)
    keep = index[:out_rows]
    obs[:len(keep)] = ref["obs"].swapaxes(1, 2).reshape(B * N, W, 6, 9, 9)[keep]
    hidden[:len(keep)] = ref["hidden"][keep]
    return obs, hidden, first, M, M_pad
