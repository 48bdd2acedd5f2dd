"""GPU: episode handling inside `rollout` at every map side and agent-count class the instance-building code serves, against
a host model made of the generator restatement (tests/generator_ref.py) and the C oracle -- no GPU twin.

When an episode ends inside the launch, the slot's next instance is built in one of three ways, and each picks its template
instances from the map side L (RW = ceil((L + 8) / 32) words per padded row, RPL = map rows per lane of a search):
* in the kernel: `regenerate_env` runs `reset_env_warp<RW, RW>` (reset() runs `<RW, ceil(L / 32)>`: they differ at L 25-32,
  57-64 and 89-96), then the heuristic-map searches, `bfs_navi_warp_pre<RW, RPL, 2>` on the slot's warp (`<4, 4, 1>` from
  L = 89) or `bfs_navi_warp` as task-queue items; a search wraps its row shuffle iff L < 16 * RPL (not at 16, 32, 48, 64, 80);
* before the launch: `pregen_reset_kernel` + `pregen_bfs_kernel` stage it with the load path's geometry, and the kernel adopts
  it by flipping the slot's heuristic-map buffer;
* beside the launch: the same staging kernels on a second stream, adopted if they are done in time.
The matrix runs each form at sides on both sides of every template switch, each with an odd agent count (the last search pair
has a dead half) and, where 8 N <= L^2 allows, one of 33-64 (two agents per lane, goals of agents 32+ in the second goal word).

Host model: each slot is an `oracle.OracleEnv` plus its episode number and step counter.  A slot that starts a step finished
(all agents on their goals after the previous step, or `steps >= cap`) loads instance env_offset + n * stride + e of the
restated generator and emits its first observation with rewards 0 (code 5), done 0, steps 0; every other slot steps the
oracle.  The model does not depend on the form, so it is built once per geometry and every form is held to it."""
import numpy as np
import pytest

from generator_ref import generate
from helpers import random_instance
from oracle import oracle

pytestmark = pytest.mark.gpu

SEED, OFFSET, STRIDE, DENSITY, CAP = 5, 1000, 4096, 0.25, 6
# every slot ends once or twice in the first call; only some end in the second, so that afterwards (staged forms) some slots
# read the second heuristic-map buffer and some the first
T1, T2 = 12, 3
RESET_SEED, RESET_OFFSET = 9, 7000
MOVES = {(-1, 0): 1, (1, 0): 2, (0, -1): 3, (0, 1): 4}   # (dx, dy) -> action
ON_GOAL, ONE_AWAY = (0, 5), (1, 6)                         # slots loaded finished / one scripted move from finishing

# (L, odd N <= 32, N in 33..64 or None where 8 N > L^2)
GEOMETRIES = [(16, 31, None), (20, 23, 49), (24, 9, 64), (25, 27, 33), (32, 31, 64), (33, 17, 47), (47, 5, 63),
              (48, 29, 64), (49, 3, 37), (56, 31, 64), (57, 11, 45), (63, 25, 64), (64, 31, 33), (72, 7, 64),
              (80, 31, 57), (81, 13, 64), (88, 1, 39), (89, 31, 64), (96, 19, 35), (97, 21, 64), (120, 31, 64)]
# form -> (mapf_debug_rollout_pregen, mapf_debug_rollout_tasks): 0 = re-generate in the kernel, 2 = stage before the launch,
# 3 = stage beside it; tasks 1 = the in-launch searches are task-queue items any warp takes
FORMS = {"inkernel": (0, 0), "inkernel_tasks": (0, 1), "before": (2, 0), "beside": (3, 1)}
CHUNKS = (0, 3)
CASES = [(L, N, form, chunk) for L, n_odd, n_wide in GEOMETRIES for N in (n_odd, n_wide) if N is not None
         for form in FORMS for chunk in CHUNKS]


def num_envs(L):
    return 24 if L <= 64 else 16


class HostSlots:
    """The rollout's episode handling, slot by slot, on the host."""

    def __init__(self, L, N, cap, seed, env_offset, stride, density, maps, starts, goals, steps):
        self.L, self.N, self.cap, self.seed, self.env_offset, self.stride, self.density = L, N, cap, seed, env_offset, stride, density
        self.envs = []
        for m, p, g in zip(maps, starts, goals):
            o = oracle.OracleEnv()
            o.load(m, p, g)
            self.envs.append(o)
        self.steps = np.array(steps, dtype=np.int32)
        self.episode = np.zeros(len(self.envs), dtype=np.int32)
        self.regenerated = 0

    def step(self, actions):
        """One rollout step -> (obs u8[B,N,6,9,9], rewards f32[B,N], codes u8[B,N], done u8[B], steps i32[B])."""
        B, N = len(self.envs), self.N
        obs = np.empty((B, N, 6, 9, 9), dtype=np.uint8)
        rew = np.zeros((B, N), dtype=np.float32)
        codes = np.empty((B, N), dtype=np.uint8)
        done = np.zeros(B, dtype=np.uint8)
        for e, o in enumerate(self.envs):
            if (o.agents_pos == o.goals_pos).all() or self.steps[e] >= self.cap:
                n = int(self.episode[e]) + 1
                m, p, g, _ = generate(self.seed, self.env_offset + n * self.stride + e, self.L, N, self.density)
                o.load(m, p, g)
                self.episode[e], self.steps[e] = n, 0
                self.regenerated += 1
                obs[e] = o.observe()[0]
                codes[e] = 5
                continue
            prev, a = o.agents_pos.copy(), actions[e]
            (ob, _), r, d, _ = o.step(a)
            obs[e], rew[e], done[e] = ob, np.asarray(r, dtype=np.float32), d
            self.steps[e] += 1
            on_goal = (prev == o.goals_pos).all(-1)
            codes[e] = np.where(a == 0, np.where(on_goal, 1, 2), np.where(rew[e] == np.float32(oracle.REWARD_FN["collision"]), 3, 0))
            if d:
                codes[e] = 4
        return obs, rew, codes, done, self.steps.copy()

    def state(self):
        return dict(map=np.stack([o.map for o in self.envs]),
                    pos=np.stack([o.agents_pos for o in self.envs]).astype(np.uint8),
                    goals=np.stack([o.goals_pos for o in self.envs]).astype(np.uint8),
                    steps=self.steps.copy(), episode=self.episode.copy(),
                    navi=np.stack([o.navi_map for o in self.envs]))


def first_instances(L, N, B, seed, env_offset, density, rng):
    """Instance env_offset + e for every slot, except that the agents of the ON_GOAL slots stand on their goals and those of
    the ONE_AWAY slots too but for one, which stands next to its goal.  -> maps, starts, goals, actions u8[B, N] that take
    that agent onto its goal (random elsewhere)."""
    maps, starts, goals = (np.stack(x) for x in zip(*[generate(seed, env_offset + e, L, N, density)[:3] for e in range(B)]))
    acts = rng.integers(0, 5, size=(B, N)).astype(np.uint8)
    for e in ON_GOAL:
        starts[e] = goals[e]
    for e in ONE_AWAY:
        starts[e] = goals[e]
        taken = {tuple(int(v) for v in g) for g in goals[e]}
        placed = False
        for a in range(N - 1, -1, -1):       # prefer the last agent: for N > 32 its goal arrives through the second goal word
            gx, gy = (int(v) for v in goals[e, a])
            for (dx, dy), act in MOVES.items():
                x, y = gx - dx, gy - dy          # stand at (x, y); action `act` moves by (dx, dy) onto the goal
                if 0 <= x < L and 0 <= y < L and maps[e, x, y] == 0 and (x, y) not in taken:
                    starts[e, a] = (x, y)
                    acts[e] = 0
                    acts[e, a] = act
                    placed = True
                    break
            if placed:
                break
        assert placed, (L, N, e)
    return maps, starts, goals, acts


class Expected:
    """Everything one geometry's runs are compared with: the two rollout calls step by step, the state after each call, the
    distance maps, a masked reset and one single-step launch afterwards."""

    def __init__(self, L, N, seed=SEED, env_offset=OFFSET, stride=STRIDE, density=DENSITY):
        B = num_envs(L)
        self.B, self.seed, self.env_offset, self.stride, self.density = B, seed, env_offset, stride, density
        rng = np.random.default_rng(L * 100 + N)
        self.maps, self.starts, self.goals, first_acts = first_instances(L, N, B, seed, env_offset, density, rng)
        # step counters staggered over [0, cap) so that the ends fall on different steps; the done-triggered slots start at 0
        self.steps0 = ((np.arange(B) * 7 + 3) % CAP).astype(np.int32)
        self.steps0[list(ON_GOAL + ONE_AWAY)] = 0
        self.actions = rng.integers(0, 5, size=(T1 + T2, B, N)).astype(np.uint8)
        self.actions[0] = first_acts
        host = HostSlots(L, N, CAP, seed, env_offset, stride, density, self.maps, self.starts, self.goals, self.steps0)
        self.out, self.after = [], []
        for t in range(T1 + T2):
            self.out.append(host.step(self.actions[t]))
            if t + 1 in (T1, T1 + T2):
                self.after.append(host.state())
        self.regenerated = host.regenerated
        self.done_ends = int(sum(o[3].sum() for o in self.out))
        self.dist = np.stack([o.dist_map for o in host.envs])
        # a masked reset of every slot but each third one, then one step of the single-step kernel
        self.reset_mask = (np.arange(B) % 3 != 1).astype(np.uint8)
        for e in np.flatnonzero(self.reset_mask):
            m, p, g, _ = generate(RESET_SEED, RESET_OFFSET + e, L, N, density)
            host.envs[e].load(m, p, g)
            host.steps[e] = 0
        self.after_reset = host.state()
        self.post_actions = rng.integers(0, 5, size=(B, N)).astype(np.uint8)
        post = [o.step(a) for o, a in zip(host.envs, self.post_actions)]
        self.post_obs = np.stack([p[0][0] for p in post]).astype(np.uint8)
        self.post_rew = np.stack([np.asarray(p[1], dtype=np.float32) for p in post])
        self.post_done = np.array([p[2] for p in post], dtype=np.uint8)
        self.post_pos = np.stack([o.agents_pos for o in host.envs]).astype(np.uint8)


_expected = {}


def expected(*key):
    """One geometry's model at a time: the cases of a geometry run one after the other."""
    if key not in _expected:
        _expected.clear()
        _expected[key] = Expected(*key)
    return _expected[key]


@pytest.fixture
def episode_form():
    """Sets the form of episode handling and the rollout's chunk for one test; restores the defaults afterwards."""
    from mapf_rl_b200 import _native
    lib = _native.lib()
    pregen0, tasks0 = lib.mapf_debug_rollout_pregen(-1), lib.mapf_debug_rollout_tasks(-1)

    def set_form(form, chunk):
        pregen, tasks = FORMS[form]
        lib.mapf_debug_rollout_pregen(pregen)
        lib.mapf_debug_rollout_tasks(tasks)
        lib.mapf_debug_rollout_tuning(1, 0, chunk, 0, -1)
    try:
        yield set_form
    finally:
        lib.mapf_debug_rollout_pregen(pregen0)
        lib.mapf_debug_rollout_tasks(tasks0)
        lib.mapf_debug_rollout_tuning(1, 0, 0, 0, 1000)


def differing(a, b):
    """Slots (leading index) where two arrays differ."""
    return np.flatnonzero((np.asarray(a) != np.asarray(b)).reshape(len(a), -1).any(1)).tolist()


def check_state(env, exp, where):
    """map, agents_pos, goals_pos, steps and navi_map of every slot against the host model's state."""
    import torch
    for name, key in (("map", "map"), ("agents_pos", "pos"), ("goals_pos", "goals"), ("steps", "steps")):
        bad = differing(getattr(env, name).cpu().numpy(), exp[key])
        assert not bad, f"{name} differs, {where}: slots {bad}"
    nv = env.navi_map
    ref = torch.as_tensor(exp["navi"]).to(nv.device)
    if not torch.equal(nv, ref):
        bad = (nv != ref).flatten(1).any(1).nonzero().flatten().tolist()
        raise AssertionError(f"navi_map differs from the oracle's heuristic maps, {where}: slots {bad}")


def run_case(env, exp, where):
    """Two rollout calls with episode handling, every step of every slot against the host model, then the state checks."""
    import torch
    B, N = exp.B, env.num_agents
    acts = torch.as_tensor(exp.actions).cuda()
    for c, (t0, t1) in enumerate(((0, T1), (T1, T1 + T2))):
        codes = torch.full((t1 - t0, B, N), 255, dtype=torch.uint8, device="cuda")
        obs, rew, done, steps = env.rollout(acts[t0:t1], out_codes=codes)
        env.check()
        obs, rew, codes, done, steps = (x.cpu().numpy() for x in (obs, rew, codes, done, steps))
        for t in range(t0, t1):
            e_obs, e_rew, e_codes, e_done, e_steps = exp.out[t]
            s = t - t0
            at = f"{where}, call {c + 1}, step {t}"
            bad = differing(obs[s], e_obs)
            assert not bad, f"observations differ, {at}: slots {bad} (reset in this step: {[e for e in bad if e_codes[e, 0] == 5]})"
            assert not differing(rew[s], e_rew), f"rewards differ, {at}: slots {differing(rew[s], e_rew)}"
            assert not differing(codes[s], e_codes), f"reward codes differ, {at}: slots {differing(codes[s], e_codes)}"
            assert np.array_equal(done[s], e_done), f"done differs, {at}: {done[s]} vs {e_done}"
            assert np.array_equal(steps[s], e_steps), f"steps differ, {at}: {steps[s]} vs {e_steps}"
        check_state(env, exp.after[c], f"{where}, after call {c + 1}")
        counts = env.episode_counts().cpu().numpy()
        assert np.array_equal(counts, exp.after[c]["episode"]), ("episode_counts", where, c + 1, counts, exp.after[c]["episode"])


def run_afterwards(env, exp, where):
    """After the calls (some slots now read the second heuristic-map buffer): distances, a masked reset, one plain step."""
    import torch
    dist = env.heuristic_distances().cpu().numpy()
    bad = differing(dist, exp.dist)
    assert not bad, f"heuristic_distances differ from the oracle's distance maps, {where}: slots {bad}"
    check_state(env, exp.after[1], f"{where}, after heuristic_distances")
    env.reset(mask=exp.reset_mask, seed=RESET_SEED, env_offset=RESET_OFFSET, density=exp.density)
    check_state(env, exp.after_reset, f"{where}, after a masked reset")
    obs, rew, done = env.step(torch.as_tensor(exp.post_actions).cuda())
    obs, rew, done = obs.cpu().numpy(), rew.cpu().numpy(), done.cpu().numpy()
    assert not differing(obs, exp.post_obs), f"step() observations differ, {where}: slots {differing(obs, exp.post_obs)}"
    assert not differing(rew, exp.post_rew) and np.array_equal(done, exp.post_done), f"step() rewards / done differ, {where}"
    assert not differing(env.agents_pos.cpu().numpy(), exp.post_pos), f"step() positions differ, {where}"
    env.check()


def make_env(exp, L, N):
    from mapf_rl_b200 import BatchedEnvironment
    env = BatchedEnvironment(exp.B, N, L)
    env.load(exp.maps, exp.starts, exp.goals)
    env.set_autoreset(CAP, seed=exp.seed, env_offset=exp.env_offset, stride=exp.stride, density=exp.density)
    env.set_state(steps=exp.steps0)
    return env


@pytest.mark.parametrize("L,N,form,chunk", CASES)
def test_rollout_episode_handling_vs_host_model(episode_form, L, N, form, chunk):
    """Two rollout calls with episode handling in one form, every step of every slot against the host model; then distances,
    a masked reset and a plain step on the state they leave."""
    exp = expected(L, N)
    # what the case is for: two episode ends per slot on average, and done-triggered ends (ON_GOAL slots at step 0, ONE_AWAY
    # slots at step 1)
    assert exp.regenerated >= 2 * exp.B and exp.done_ends >= len(ONE_AWAY)
    assert all(exp.out[0][2][e, 0] == 5 for e in ON_GOAL) and all(exp.out[1][2][e, 0] == 5 for e in ONE_AWAY)
    episode_form(form, chunk)
    env = make_env(exp, L, N)
    where = f"L {L}, N {N}, {form}, chunk {chunk}"
    run_case(env, exp, where)
    run_afterwards(env, exp, where)
    env.close()


@pytest.mark.parametrize("form", list(FORMS))
def test_rollout_episode_handling_64bit_instance_index(episode_form, form):
    """env_offset + n * stride + e crosses 2^32 inside the launch (n = 2), with a seed above 2^32 and drawn densities."""
    L, N = 33, 17
    B = num_envs(L)
    exp = expected(L, N, 2**32 + 0x5EED, 2**32 - 2 * B, B, None)
    assert exp.after[0]["episode"].max() >= 2
    episode_form(form, 3)
    env = make_env(exp, L, N)
    where = f"64-bit index, {form}"
    run_case(env, exp, where)
    run_afterwards(env, exp, where)
    env.close()


@pytest.mark.parametrize("L", range(2, 121))
def test_load_heuristic_maps_every_side(L):
    """load() at every side 2-120 (`bfs_navi_kernel` at every geometry it is compiled for): heuristic maps, and distances with
    the same maps recomputed, against the oracle on instances with unreachable cells (starts and goals in any component)."""
    import torch
    from mapf_rl_b200 import BatchedEnvironment
    rng = np.random.default_rng(L)
    B, N = 3, int(rng.integers(1, min(64, L * L // 2) + 1))
    insts = [random_instance(rng, L, N, 0.3) for _ in range(B)]
    maps, starts, goals = (np.stack(x) for x in zip(*insts))
    env = BatchedEnvironment(B, N, L)
    env.load(maps, starts, goals)
    ref = [oracle.navi(m, g) for m, g in zip(maps, goals)]
    nv_ref = torch.as_tensor(np.stack([r[1] for r in ref])).cuda()
    dist_ref = np.stack([r[0] for r in ref])
    assert torch.equal(env.navi_map, nv_ref), (L, N, (env.navi_map != nv_ref).flatten(1).any(1).nonzero().flatten().tolist())
    dist = env.heuristic_distances().cpu().numpy()
    assert not differing(dist, dist_ref), (L, N, differing(dist, dist_ref))
    dist = env.heuristic_distances(env_ids=[2, 0]).cpu().numpy()
    assert np.array_equal(dist, dist_ref[[2, 0]]), (L, N)
    assert torch.equal(env.navi_map, nv_ref), (L, N)
    env.close()
