"""The kinematic step kernel's fragment schedule: tile outer, step inner, joint warps one work item ahead of the task warp.

Within a rollout fragment (pnr_step_many) a CTA runs every step on a tile before it takes the next one.  The joint warps
integrate step s + 1 of an env while the task warp is still finishing step s, so the one dependency between the two steps,
an auto-reset decided by the task warp, travels through shared memory: a `reached` reset is only known after the task
warp's forward kinematics.  These cases make such resets the common case and cover the schedule's edges:

  1. done_distance at the median start distance, so that a good share of the envs (about one in eight) reach their
     target in a step and reset; TimeLimit off, and TimeLimit 1 (every step resets every env, reached or truncated).  Fragment lengths 1, 2, 3,
     8, 17; sizes with one tile per CTA (4,096 and 16,384 envs), fewer than 32 envs, and ragged tails whose last tile
     is streamed without a bulk copy.  Fragments equal single steps bit for bit: observations, rewards, flags, state,
     boxes and episode statistics.
  2. The same with obstacles and a per-env box redrawn at every reset, both observation modes, and against the C oracle.
  3. Fragments captured in a CUDA graph and replayed back to back (programmatic dependent launch between them) equal a
     graph of single steps."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle.c_oracle import COracleBatch
from oracle.reach_oracle import OracleChain, OracleConfig
from tests.test_gpu_parity import check_obs

pytestmark = pytest.mark.gpu

STATE_KEYS = ("r", "v", "a", "potential", "target", "t", "ep_return")
STAT_KEYS = ("episodes", "sum_length", "env_steps", "reached_target", "max_return", "min_return")
_DISTANCE = {}


def reach_distance():
    """The median distance of a freshly reset env to its target, used as done_distance."""
    if "d" not in _DISTANCE:
        from pioneer_b200 import BatchedPioneerEnv
        probe = BatchedPioneerEnv(4096, seed=0)
        _DISTANCE["d"] = float(probe.observe()[:, 135].median())
        probe.close()
    return _DISTANCE["d"]


def make_env(n, limit, obstacles=False, obs_mode="terminal", seed=0):
    from pioneer_b200 import BatchConfig, BatchedPioneerEnv, PioneerKinematicConfig, demo_obstacles
    bc = BatchConfig(max_episode_steps=limit, auto_reset=True, obs_mode=obs_mode,
                     obstacles=demo_obstacles() if obstacles else [], contact_penalty=0.5 if obstacles else 0.0,
                     random_box=obstacles)
    return BatchedPioneerEnv(n, seed=seed, batch_config=bc, pioneer_config=PioneerKinematicConfig(done_distance=reach_distance()))


def make_oracle(env, seed):
    bc = env.batch_config
    cfg = OracleConfig(max_episode_steps=bc.max_episode_steps, done_distance=reach_distance(), contact_penalty=bc.contact_penalty,
                       obstacles=tuple((o.kind, o.position, o.extent) for o in bc.obstacles),
                       random_box=(bc.box_pos_lo, bc.box_pos_hi, bc.box_size_lo, bc.box_size_hi) if bc.random_box else None)
    return COracleBatch(OracleChain.from_model(env.chain), env.n_envs, cfg, arith="np2", seed=seed, obs_mode=bc.obs_mode)


def buffers(T, n):
    n_pad = (n + 3) // 4 * 4                      # every obs[t] on a 16-byte boundary
    return (torch.empty((T, n_pad, 137), device="cuda")[:, :n], torch.empty((T, n), device="cuda"),
            torch.empty((T, n), dtype=torch.uint8, device="cuda"))


def reached_resets(flags):
    """Episodes that ended because the target was reached (done, not truncated by the TimeLimit)."""
    f = flags.to(torch.int32)
    return int(((f & 1) != 0).logical_and((f & 2) == 0).sum())


def assert_same_envs(a, b, what):
    sa, sb = a.state(), b.state()
    for key in STATE_KEYS:
        assert torch.equal(sa[key], sb[key]), (what, key)
    if a.batch_config.random_box:
        assert torch.equal(a.boxes(), b.boxes()), what


def assert_same_stats(a, b):
    st_a, st_b = a.episode_stats(), b.episode_stats()
    for key in STAT_KEYS:
        assert st_a[key] == st_b[key], (key, st_a[key], st_b[key])
    for key in ("sum_return", "sum_return_sq"):   # float64 atomics, added in an order that depends on the launch shape
        assert abs(st_a[key] - st_b[key]) <= 1e-9 * abs(st_b[key]), (key, st_a[key], st_b[key])
    return st_a


def fragments_vs_single_steps(n, T, limit, obstacles=False, obs_mode="terminal", fragments=3, seed=0):
    """Twin envs: `a` runs fragments of T steps in one launch, `b` the same actions one step per launch."""
    a, b = (make_env(n, limit, obstacles, obs_mode, seed=seed) for _ in range(2))
    g = torch.Generator(device="cuda").manual_seed(seed + 1)
    lo, hi = torch.as_tensor(a.action_space.low).cuda(), torch.as_tensor(a.action_space.high).cuda()
    obs, rew, flg = buffers(T, n)
    reached = 0
    for k in range(fragments):
        act = lo + torch.rand((T, n, 6), device="cuda", generator=g) * (hi - lo)
        a.step_many(act, obs, rew, flg)
        for t in range(T):
            o, r, f = b.step_tensor(act[t])
            assert torch.equal(f, flg[t]), (k, t, int((f != flg[t]).sum()))
            assert torch.equal(r, rew[t]), (k, t, float((r - rew[t]).abs().max()))
            assert torch.equal(o, obs[t]), (k, t, float((o - obs[t]).abs().max()))
        assert_same_envs(a, b, k)
        reached += reached_resets(flg)
    st = assert_same_stats(a, b)
    a.close(); b.close()
    return reached, st


SIZES = [4096, 16384, 29, 4096 + 37, 1000 + 2]


# ---------------------------------------------------------------------------------------------
# 1. distance resets inside fragments, every fragment length, sizes at the schedule's edges
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("T", [1, 2, 3, 8, 17])
@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("limit", [0, 1])
def test_distance_resets_fragments_equal_single_steps(limit, n, T):
    reached, st = fragments_vs_single_steps(n, T, limit, fragments=2 if T > 8 else 3)
    steps = (2 if T > 8 else 3) * T
    assert reached >= n * steps // 20, (reached, n * steps)     # `reached` resets are common, not a corner case
    if limit == 1:
        assert st["episodes"] == n * steps                         # consecutive resets of the same env, every step
    assert st["reached_target"] == reached


# ---------------------------------------------------------------------------------------------
# 2. obstacles + per-env box redrawn at every reset; the C oracle
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("T", [2, 3, 17])
@pytest.mark.parametrize("obs_mode", ["terminal", "autoreset"])
@pytest.mark.parametrize("n", [4096, 29, 4096 + 37])
def test_distance_resets_with_random_boxes_fragments_equal_single_steps(n, obs_mode, T):
    reached, _ = fragments_vs_single_steps(n, T, 0, obstacles=True, obs_mode=obs_mode, fragments=2, seed=5)
    assert reached >= n * 2 * T // 20, reached


@pytest.mark.parametrize("obstacles", [False, True])
@pytest.mark.parametrize("limit", [0, 1, 3])
@pytest.mark.parametrize("n,T", [(16384, 8), (4096 + 37, 17), (29, 3)])
def test_distance_reset_fragments_vs_c_oracle(n, T, limit, obstacles):
    """Flags and rewards of every step, the last observation, state and boxes of every fragment against the C oracle."""
    seed = 12
    env = make_env(n, limit, obstacles, seed=seed)
    orc = make_oracle(env, seed)
    rng = np.random.default_rng(seed)
    obs, rew, flg = buffers(T, n)
    worst, reached = 0.0, 0
    for k in range(3):
        act = (rng.uniform(-1, 1, size=(T, n, 6)) * env.a_max).astype(np.float32)
        env.step_many(torch.as_tensor(act).cuda(), obs, rew, flg)
        rew_h, flg_h = rew.cpu().numpy(), flg.cpu().numpy()
        for t in range(T):
            o_obs, o_rew, o_flags = orc.step(act[t], want_obs=(t == T - 1))
            assert np.array_equal(flg_h[t], o_flags), (k, t, int((flg_h[t] != o_flags).sum()))
            worst = max(worst, float(np.abs(rew_h[t] - o_rew).max()))
        check_obs(obs[T - 1].cpu().numpy(), o_obs, f"fragment {k}")
        s, o = env.state(), orc.state()
        for key in ("r", "v", "a", "t"):
            assert np.array_equal(s[key].cpu().numpy(), o[key]), (k, key)
        assert np.array_equal(s["target"].cpu().numpy(), o["target"].astype(np.float32)), k
        if obstacles:
            assert np.array_equal(env.boxes().cpu().numpy().astype(np.float64), orc.boxes()), k
        reached += reached_resets(flg)
    assert worst <= 2e-3, worst
    assert reached >= n * 3 * T // 20, reached
    st = env.episode_stats()
    assert st["episodes"] == orc.stats[0] and st["sum_length"] == orc.stats[2] and st["reached_target"] == orc.stats[7]
    env.close()


# ---------------------------------------------------------------------------------------------
# 3. fragments replayed from a CUDA graph, back to back
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [16384 + 5, 4096])
def test_graph_fragments_back_to_back_equal_graph_single_steps(n):
    """Graph A: the reset-counter advance, then two fragments of 8 steps, two step kernels in a row (with programmatic
    dependent launch on these sizes the second may start while the first drains).  Graph B on a twin: the same advance and
    16 single steps.  Both are their handle's first graph and capture at the same call counter, so they draw the same
    reset keys: three replays each must agree bit for bit."""
    T = 8
    a, b = (make_env(n, 0, seed=3) for _ in range(2))
    g = torch.Generator(device="cuda").manual_seed(7)
    lo, hi = torch.as_tensor(a.action_space.low).cuda(), torch.as_tensor(a.action_space.high).cuda()
    act = lo + torch.rand((2 * T, n, 6), device="cuda", generator=g) * (hi - lo)
    obs_a, rew_a, flg_a = buffers(2 * T, n)
    obs_b, rew_b, flg_b = buffers(2 * T, n)
    a.step_many(act[:T], obs_a[:T], rew_a[:T], flg_a[:T])         # eager warm-up (kernel attributes), mirrored on the twin
    for t in range(T):
        b.step_tensor(act[t], out=(obs_b[t], rew_b[t], flg_b[t]))
    torch.cuda.synchronize()
    assert torch.equal(obs_a[:T], obs_b[:T]) and torch.equal(flg_a[:T], flg_b[:T])
    ga, gb = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
    with torch.cuda.graph(ga):
        a.advance_reset_counter(2 * T)
        a.step_many(act[:T], obs_a[:T], rew_a[:T], flg_a[:T])
        a.step_many(act[T:], obs_a[T:], rew_a[T:], flg_a[T:])
    with torch.cuda.graph(gb):
        b.advance_reset_counter(2 * T)
        for t in range(2 * T):
            b.step_tensor(act[t], out=(obs_b[t], rew_b[t], flg_b[t]))
    reached = 0
    for k in range(3):
        ga.replay(); gb.replay()
        torch.cuda.synchronize()
        assert torch.equal(flg_a, flg_b), k
        assert torch.equal(rew_a, rew_b), k
        assert torch.equal(obs_a, obs_b), k
        assert_same_envs(a, b, k)
        reached += reached_resets(flg_a)
    assert reached >= n * 3 * 2 * T // 20, reached
    assert_same_stats(a, b)
    a.close(); b.close()
