"""The prioritized-replay sum tree against the oracle on the call stream the replay store makes, at the store's sizes.

`tests/test_gpu_per.py` checks the tree's kernels on synthetic batches.  Here every call the actor and the learner make is
replayed on a device `SumTree` and on `oracle.OracleSumTree` side by side, and after every call the device heap must equal
the oracle's bit for bit:
  * evict (BatchedActor._take_slots): k*S leaves of k ring slots set to 0;
  * publish (BatchedActor._finish): the k*S leaves of those slots in one update, td**alpha for a random episode size and 0
    past it, in ring order (unsorted where the ring wraps) or in environment order (slots permuted);
  * learner cycle (learner.py): the fused TD update on the indices of the previous sample, with the stale-slot window
    [old_ptr, ptr), then the next sample with its importance weights.
The batch sizes cross every threshold where the kernels change path (n <= 256 sorted, <= 4096, > 4096), at capacities
2^18 (bench_c5: 4096 slots x 64), 2^19 (the reference: 2048 x 256), 2^20 and 2^21 (the sampler's last group has 1 and 2
levels), 2^22 (8192 environments) and 2^24 (update shared memory past 48 KB).

The sampler is also driven at its edges (u = 0, u = nextafter(1, 0), batches past one CTA's threads, trees that are empty,
all equal, or nonzero at one leaf only), and a sample that lands on a leaf of priority 0 -- which the reference rejects
with an assert (buffer.py:74) -- must make `SumTree.check()` raise AssertionError while returning the reference's leaf.
Last, the real BatchedActor and BatchedLearner run at bench_c5's per-GPU shape with every tree call mirrored into the
oracle.
"""
import numpy as np
import pytest

from oracle import oracle

ALPHA, BETA = 0.6, 0.4
TOP = np.nextafter(1.0, 0.0)   # the largest uniform below 1
DEV = "cuda:0"


# ---- trees built on the host ------------------------------------------------------------------------------------------
def heap_of(leaves: np.ndarray) -> np.ndarray:
    """The array heap buffer.py:25 holds for these leaves: every parent = left + right (fp64), level by level."""
    cap = leaves.shape[0]
    t = np.zeros(2 * cap - 1)
    t[cap - 1:] = leaves
    start, width = cap - 1, cap
    while width > 1:
        width //= 2
        p = (start - 1) // 2
        t[p:p + width] = t[start:start + 2 * width:2] + t[start + 1:start + 2 * width:2]
        start = p
    return t


def episode_leaves(rng, S):
    """Leaves of one published episode: td**alpha over a random size in 1..S-1 with some exact-zero TDs, then 0."""
    size = int(rng.integers(1, S))
    td = rng.exponential(1.0, S)
    td[rng.random(S) < 0.05] = 0.0
    td[size:] = 0.0
    return td ** ALPHA


def blocky_leaves(cap, seed, S=256):
    """A store filled part way: about 70% of the first half of the slots hold an episode, the right half is empty."""
    rng = np.random.default_rng(seed)
    S = min(S, cap)
    leaves = np.zeros(cap)
    for s in range(max(1, cap // S // 2)):
        if rng.random() < 0.7:
            leaves[s * S:(s + 1) * S] = episode_leaves(rng, S) if S > 1 else rng.random()
    return leaves


def edge_trees(cap):
    """name -> leaves of the sampler-edge trees."""
    one = lambda i: np.where(np.arange(cap) == i, 0.75, 0.0)
    return {"blocky": blocky_leaves(cap, 1), "zero": np.zeros(cap), "left": one(0), "right": one(cap - 1),
            "middle": one(cap // 2), "equal": np.ones(cap)}


def test_zero_leaf_constructions_sample_priority_zero():
    """The premise of the latch tests, on the CPU: the oracle's descent (buffer.py:56-78) does end on a leaf of priority 0
    for an empty tree, and for a partly filled 2^19 store whose last stratum, p = 191*iv + u*iv with u = nextafter(1, 0),
    rounds up to the sum of the filled leaves: the descent passes them and ends on an empty leaf."""
    cap, B = 1 << 19, 192
    ref = oracle.OracleSumTree(cap)
    leaves = np.arange(cap, dtype=np.int64)
    ref.batch_update(leaves.copy(), blocky_leaves(cap, 1))
    assert np.array_equal(ref.tree, heap_of(blocky_leaves(cap, 1)))   # the host heap is the oracle's
    for seed in (1, 2):
        ref.tree[:] = heap_of(blocky_leaves(cap, seed))
        idx, pr = ref.batch_sample(B, np.full(B, TOP))
        assert pr[-1] == 0.0 and (pr[:-1] > 0).all(), seed
        idx, pr = ref.batch_sample(B, np.random.default_rng(seed).random(B))
        assert (pr > 0).all()
    ref.tree[:] = 0.0
    idx, pr = ref.batch_sample(B, np.full(B, 0.5))
    assert (pr == 0.0).all()


# ---- a device tree and its oracle shadow ------------------------------------------------------------------------------
class Shadow:
    """A device SumTree and an OracleSumTree that receive the same calls; every call is checked against the oracle."""

    def __init__(self, tree, cap):
        self.tree, self.cap = tree, cap
        self.ref = oracle.OracleSumTree(cap)

    def set_leaves(self, leaves):
        import torch
        self.tree.update_device(torch.arange(self.cap, dtype=torch.int64, device=DEV), torch.as_tensor(leaves).to(DEV))
        self.ref.tree[:] = heap_of(leaves)
        self.heap_equal("set_leaves")

    def heap_equal(self, what):
        import torch
        want = torch.from_numpy(self.ref.tree).to(DEV)
        got = self.tree.tree
        if not torch.equal(got, want):
            node = int((got != want).nonzero()[0, 0])
            pytest.fail(f"{what}: the device heap differs from the oracle's first at node {node} (depth "
                        f"{(node + 1).bit_length() - 1} of {self.ref.layer - 1}): {float(got[node])!r} != {float(want[node])!r}")

    def update(self, idx, prio, what):
        """SumTree.update_device of leaves idx int64[n] = prio float64[n] (host arrays)."""
        import torch
        self.tree.update_device(torch.as_tensor(idx).to(DEV), torch.as_tensor(prio).to(DEV))
        self.ref.batch_update(np.array(idx, dtype=np.int64), np.asarray(prio, dtype=np.float64))
        self.tree.check()
        self.heap_equal(what)

    def check_sample(self, idx, prio, weights, u, what, allow_zero=True):
        """Device sample (CUDA tensors) against the oracle's descent on the same uniforms; the latch against its priorities."""
        B = int(u.shape[0])
        ri, rp = self.ref.batch_sample(B, u)
        gi, gp = idx.cpu().numpy(), prio.cpu().numpy()
        bad = np.flatnonzero((gi != ri) | (gp.view(np.uint64) != rp.view(np.uint64)))
        assert bad.size == 0, (f"{what}: sample {bad[0]} of {B} (u = {u[bad[0]]!r}): device leaf {gi[bad[0]]} priority "
                               f"{gp[bad[0]]!r}, oracle leaf {ri[bad[0]]} priority {rp[bad[0]]!r}")
        zero = not (rp > 0).all()
        if weights is not None and not zero:
            np.testing.assert_allclose(weights.cpu().numpy(), np.power(rp / rp.min(), -BETA), rtol=1e-6, atol=0, err_msg=what)
        if zero:
            assert allow_zero, f"{what}: sampled a leaf of priority 0 ({int((rp <= 0).sum())} of {B})"
            with pytest.raises(AssertionError):
                self.tree.check()
        self.tree.check()   # the latch is cleared, and nothing else was latched
        return zero

    def after_cycle(self, out, update, u, old_ptr, ptr, slot_steps, what, alpha=ALPHA, allow_zero=True):
        """Checks of one SumTree.cycle call, whose results are in `out`: the TD update half against worker.py:300-308 and
        the oracle tree, then the sample half.  The device evaluates pow(fp32 priority, alpha) with CUDA's pow, within 2 ulp
        of numpy's: the updated leaves are checked at 1e-15 relative and the device's values then written into the oracle
        too, so that everything after them stays bit-comparable."""
        import torch
        if update is not None:
            ix = update["idx"].cpu().numpy()
            host = {k: update[k].cpu().numpy() for k in ("q_online", "q_target_next", "action", "reward", "done", "steps")}
            td, pr = oracle.learner_td(host["q_online"], host["q_target_next"], host["action"], host["reward"], host["done"],
                                       host["steps"])
            np.testing.assert_allclose(out["prio"].cpu().numpy(), pr, rtol=1e-5, atol=1e-7, err_msg=what)
            gpr = out["prio"].cpu().numpy().astype(np.float64)
            if ptr > old_ptr:    # worker.py:192-201
                keep = (ix < old_ptr * slot_steps) | (ix >= ptr * slot_steps)
            elif ptr < old_ptr:
                keep = (ix < old_ptr * slot_steps) & (ix >= ptr * slot_steps)
            else:
                keep = np.ones(ix.shape[0], dtype=bool)
            kix, kpr = ix[keep], gpr[keep]
            if kix.size:
                uniq, pos = np.unique(kix[::-1], return_index=True)   # the last duplicate wins (buffer.py:97)
                want = np.power(kpr[kix.size - 1 - pos], alpha)
                got = self.tree.tree[torch.as_tensor(uniq, device=DEV) + (self.cap - 1)].cpu().numpy()
                np.testing.assert_allclose(got, want, rtol=1e-15, atol=0, err_msg=what)
                self.ref.batch_update(uniq.copy(), got)
            self.heap_equal(what + " (update half)")
        if u is not None:
            return self.check_sample(out["idx"], out["sample_prio"], out["weights"], u, what + " (sample half)",
                                     allow_zero=allow_zero)
        return False


def learner_batch(rng, idx):
    """The update half of a learner cycle for the given leaf indices (int64 CUDA tensor)."""
    import torch
    n = int(idx.numel())
    cuda = lambda a: torch.as_tensor(a).to(DEV).contiguous()
    return dict(q_online=cuda(rng.normal(size=(n, 5)).astype(np.float32)),
                q_target_next=cuda(rng.normal(size=(n, 5)).astype(np.float32)),
                action=cuda(rng.integers(0, 5, size=n)),
                reward=cuda(rng.choice([-0.075, -0.5, 0.0, 3.0], size=n).astype(np.float32)),
                done=cuda((rng.random(n) < 0.1).astype(np.float32)),
                steps=cuda(rng.integers(1, 3, size=n).astype(np.float32)),
                idx=idx.contiguous())


# ---- (a) the store's call stream --------------------------------------------------------------------------------------
class StoreStream:
    """The tree calls of a replay store with `slots` episode slots of S steps, driven by a schedule of operations."""

    def __init__(self, slots, S, seed, start_slot):
        from mapf_rl_b200 import SumTree
        self.slots, self.S, self.cap = slots, S, slots * S
        self.rng = np.random.default_rng(seed)
        self.sh = Shadow(SumTree(self.cap, device=DEV), self.cap)
        self.ptr = start_slot % slots   # the ring pointer (ReplayStore.ptr)
        self.evicted = []               # slot batches taken and not yet published
        self.last = None                # (sampled indices, ptr at sampling time) of the previous cycle
        self.samples = 0

    def leaves_of(self, slots):
        return (np.asarray(slots, dtype=np.int64)[:, None] * self.S + np.arange(self.S)[None, :]).reshape(-1)

    def evict(self, k):
        slots = (self.ptr + np.arange(k)) % self.slots
        self.ptr = (self.ptr + k) % self.slots
        self.evicted.append(slots)
        leaves = self.leaves_of(slots)
        self.sh.update(leaves, np.zeros(leaves.shape[0]), f"evict {k} slots from {slots[0]}")

    def publish(self, order):
        slots = self.evicted.pop(0)
        if order == "env":   # the environments that finish together took their slots at different times
            slots = self.rng.permutation(slots)
        prio = np.concatenate([episode_leaves(self.rng, self.S) for _ in slots])
        self.sh.update(self.leaves_of(slots), prio, f"publish {len(slots)} slots in {order} order")

    def window(self, n, where):
        """n consecutive leaves, at the ring pointer or across the end of the tree: the thresholds n = k*S cannot hit."""
        start = self.ptr * self.S if where == "ring" else self.cap - n // 2
        leaves = (start + np.arange(n)) % self.cap
        prio = np.concatenate([episode_leaves(self.rng, self.S) for _ in range(-(-n // self.S))])[:n]
        self.sh.update(leaves.astype(np.int64), prio, f"update of {n} leaves ({where})")

    def cycle(self, n_sample):
        import torch
        update = old_ptr = None
        if self.last is not None:
            idx, old_ptr = self.last
            update = learner_batch(self.rng, idx)
        self.samples += 1
        u = np.full(n_sample, TOP) if self.samples % 4 == 0 else self.rng.random(n_sample)
        out = self.sh.tree.cycle(update=update, sample_size=n_sample, uniforms=torch.as_tensor(u).to(DEV), beta=BETA,
                                 old_ptr=old_ptr or 0, ptr=self.ptr, slot_steps=self.S, alpha=ALPHA)
        self.sh.after_cycle(out, update, u, old_ptr, self.ptr, self.S,
                            f"cycle: update {0 if update is None else int(update['idx'].numel())}, sample {n_sample}")
        self.last = (out["idx"].clone(), self.ptr)

    def run(self, schedule):
        for op, *args in schedule:
            getattr(self, op)(*args)


# S = 64 (bench_c5): n = k*S = 64, 256 (wrapping the ring), 320, 4096, 4160 and 131072, plus 255 / 257 / 4097 leaves;
# learner updates of 192, 255, 256, 257 and 1000 entries
SCHEDULE_S64 = [
    ("evict", 4), ("publish", "ring"), ("evict", 64), ("publish", "ring"), ("cycle", 192), ("cycle", 192),
    ("evict", 1), ("cycle", 255), ("publish", "ring"), ("cycle", 192),
    ("evict", 5), ("publish", "env"), ("evict", 4), ("publish", "env"), ("cycle", 256), ("cycle", 257), ("cycle", 1000),
    ("cycle", 192), ("window", 255, "end"), ("window", 257, "ring"), ("window", 4097, "end"), ("window", 64, "ring"),
    ("evict", 65), ("publish", "env"), ("cycle", 192), ("evict", 2048), ("cycle", 192), ("publish", "env"), ("cycle", 192),
    ("evict", 2048), ("publish", "ring"), ("cycle", 192), ("cycle", 192),
]
# S = 256: n = 256, 512 (wrapping), 768, 4096 and 4352, plus 64 / 255 / 257 / 4097 leaves
SCHEDULE_S256 = [
    ("evict", 2), ("publish", "ring"), ("evict", 16), ("publish", "ring"), ("cycle", 192), ("evict", 1), ("cycle", 192),
    ("publish", "ring"), ("evict", 3), ("publish", "env"), ("cycle", 256), ("cycle", 257), ("cycle", 1000), ("cycle", 192),
    ("window", 255, "end"), ("window", 257, "ring"), ("window", 4097, "end"), ("window", 64, "ring"),
    ("evict", 17), ("publish", "env"), ("cycle", 192), ("cycle", 192), ("cycle", 192),
]
# 2^24 leaves: the 256-entry updates need more than 48 KB of shared memory
SCHEDULE_SHORT = [
    ("evict", 1), ("publish", "ring"), ("evict", 16), ("publish", "ring"), ("evict", 2), ("publish", "env"),
    ("cycle", 256), ("cycle", 256), ("cycle", 192),
]


@pytest.mark.gpu
@pytest.mark.parametrize("slots,S,schedule", [
    (4096, 64, SCHEDULE_S64),       # 2^18, bench_c5 (2048 environments, episode cap 64)
    (2048, 256, SCHEDULE_S256),     # 2^19, the reference (train.py:21, config.py:29)
    (4096, 256, SCHEDULE_S256),     # 2^20: the sampler's last group is one level
    (8192, 256, SCHEDULE_S256),     # 2^21: the sampler's last group is two levels
    (16384, 256, SCHEDULE_S256),    # 2^22, 8192 environments
    (65536, 256, SCHEDULE_SHORT),   # 2^24
], ids=["2^18", "2^19", "2^20", "2^21", "2^22", "2^24"])
def test_store_call_stream_vs_oracle(slots, S, schedule):
    """The ring starts two slots before its end, so the first small publish wraps: an unsorted batch of <= 256 leaves."""
    StoreStream(slots, S, seed=slots + S, start_slot=slots - 2).run(schedule)


# ---- (b) the sampler's edges ------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("cap", [1 << 10, 1 << 12, 1 << 19, 1 << 20, 1 << 21])
def test_sampler_edges_vs_oracle(cap):
    """2^10: the whole tree in shared memory; 2^12: one 2-level group below it; 2^19: three 3-level groups; 2^20 and 2^21:
    a last group of one and two levels.  Batches past 256 samples take the strided loop and the minimum across warps.
    With u = 0 on the all-equal tree every prefix falls on a node boundary (the `p <= left` tie goes left)."""
    import torch
    from mapf_rl_b200 import SumTree
    sh = Shadow(SumTree(cap, device=DEV), cap)
    rng = np.random.default_rng(cap)
    stale = torch.arange(192, dtype=torch.int64, device=DEV)   # update entries the stale window [0, 1) masks out
    zeros = 0
    for name, leaves in edge_trees(cap).items():
        sh.set_leaves(leaves)
        for B in (1, 192, 255, 256, 257, 1000, 4096):
            for uname, u in (("0", np.zeros(B)), ("top", np.full(B, TOP)), ("random", rng.random(B))):
                what = f"tree {name}, batch {B}, u {uname}"
                ud = torch.as_tensor(u).to(DEV)
                gi, gp, gw = sh.tree.sample_device(B, ud, beta=BETA)
                zero = sh.check_sample(gi, gp, gw, u, what + ", sample_device")
                out = sh.tree.cycle(sample_size=B, uniforms=ud, beta=BETA)
                assert sh.check_sample(out["idx"], out["sample_prio"], out["weights"], u, what + ", cycle") == zero
                # update + sample in one launch; every update entry is stale, so the tree stays as built while the sample
                # reads the top of the tree the update left in shared memory
                upd = learner_batch(rng, stale)
                out = sh.tree.cycle(update=upd, sample_size=B, uniforms=ud, beta=BETA, old_ptr=0, ptr=1, slot_steps=cap)
                assert sh.after_cycle(out, upd, u, 0, 1, cap, what + ", update + sample cycle") == zero
                zeros += zero
        sh.heap_equal(f"tree {name}")
    assert zeros > 0   # the empty tree at least


# ---- (c) the latch -----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("first", ["index", "priority"])
def test_index_and_priority_latches_are_reported_one_per_call(first):
    """An out-of-range leaf index and a sample of priority 0 latched together: check() raises IndexError and
    AssertionError in two successive calls, each naming its own condition, and the third call passes."""
    import torch
    from mapf_rl_b200 import SumTree
    cap = 1 << 10
    t = SumTree(cap, device=DEV)   # all leaves 0
    u = torch.full((8,), 0.5, dtype=torch.float64, device=DEV)

    def bad_index():
        t.update_device(torch.as_tensor([3, cap + 5], device=DEV), torch.zeros(2, dtype=torch.float64, device=DEV))

    def zero_sample():
        idx, pr, _ = t.sample_device(8, u)
        assert (pr == 0).all()

    for f in ((bad_index, zero_sample) if first == "index" else (zero_sample, bad_index)):
        f()
    raised = []
    for _ in range(2):
        with pytest.raises((IndexError, AssertionError)) as e:
            t.check()
        raised.append(e.type)
        assert ("leaf index outside" in str(e.value)) == (e.type is IndexError), str(e.value)
    assert set(raised) == {IndexError, AssertionError}
    t.check()


# ---- (d) the real actor and learner, shadowed -------------------------------------------------------------------------
@pytest.mark.gpu
def test_actor_and_learner_tree_calls_vs_oracle():
    """BatchedActor at bench_c5's per-GPU shape (2048 environments on 40x40 boards, episode cap 64: 4096 slots, 2^18
    leaves; 8 agents instead of 32, the tree traffic does not depend on it), then BatchedLearner updates between actor
    steps.  Every update_device and cycle call of the store's tree is mirrored into the oracle with the uniforms the
    learner drew, and checked as in the call-stream test; no sample may land on a leaf of priority 0."""
    import torch
    from mapf_rl_b200 import BatchedEnvironment, ReplayStore
    from mapf_rl_b200.actor import BatchedActor
    from mapf_rl_b200.learner import BatchedLearner
    from mapf_rl_b200.qnet import Network
    torch.manual_seed(0)
    B, N, L, cap = 2048, 8, 40, 64
    env = BatchedEnvironment(B, N, L, device=DEV)
    net = Network().to(DEV)
    store = ReplayStore(4096, max_num_agents=N, device=DEV, max_steps=cap)
    tree = store.priority_tree
    assert tree.capacity == 1 << 18
    sh = Shadow(tree, tree.capacity)
    calls = {"update": 0, "cycle": 0, "sizes": set()}
    update_device, cycle = tree.update_device, tree.cycle

    def mirrored_update(idx, prio):
        update_device(idx, prio)
        ix = torch.as_tensor(idx, dtype=torch.int64).cpu().numpy()
        sh.ref.batch_update(ix.copy(), torch.as_tensor(prio, dtype=torch.float64).cpu().numpy())
        calls["update"] += 1
        calls["sizes"].add(int(ix.shape[0]))
        sh.heap_equal(f"actor update {calls['update']} of {ix.shape[0]} leaves")

    def mirrored_cycle(update=None, sample_size=0, uniforms=None, beta=None, old_ptr=0, ptr=0, slot_steps=cap, gamma=0.99,
                       alpha=ALPHA, out=None):
        assert uniforms is not None and beta is not None
        u = uniforms.cpu().numpy().copy()   # the learner's own draw
        res = cycle(update=update, sample_size=sample_size, uniforms=uniforms, beta=beta, old_ptr=old_ptr, ptr=ptr,
                    slot_steps=slot_steps, gamma=gamma, alpha=alpha, out=out)
        calls["cycle"] += 1
        sh.after_cycle(res, update, u if sample_size else None, old_ptr, ptr, slot_steps, f"learner cycle {calls['cycle']}",
                       alpha=alpha, allow_zero=False)
        return res

    tree.update_device, tree.cycle = mirrored_update, mirrored_cycle
    actor = BatchedActor(env, net, store, epsilon=0.3, seed=3, density=0.3, max_steps=cap)
    # the environments start together and almost all of them run to the cap: episodes end in waves every `cap` steps.  The
    # learner's updates straddle the fourth wave, so the ring moves between a batch's draw and its update (stale window)
    actor.run(4 * cap - 10)
    learner = BatchedLearner(net, store, seed=7)
    assert learner.ready(4 * learner.batch_size)
    ptr0 = store.ptr
    for it in range(20):
        actor.step()
        stats = learner.update(want_stats=it == 19)
    assert store.ptr != ptr0
    assert np.isfinite(stats["loss"])
    tree.check()
    env.check()
    assert calls["cycle"] == 21 and max(calls["sizes"]) > 4096, calls
