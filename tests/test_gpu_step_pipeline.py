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
import pytest

torch = pytest.importorskip("torch")

from tests._gpu import (assert_same_envs, assert_same_stats, fragment_buffers, fragments_equal_single_steps,
                        k1_fragments_vs_c_oracle, kinematic_env, reached_resets, uniform_actions)

pytestmark = pytest.mark.gpu

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
    return kinematic_env(n, max_episode_steps=limit, obstacles=obstacles, obs_mode=obs_mode, done_distance=reach_distance(),
                         seed=seed)


def fragments_vs_single_steps(n, T, limit, obstacles=False, obs_mode="terminal", fragments=3, seed=0):
    """Twin envs: `a` runs fragments of T steps in one launch, `b` the same actions one step per launch."""
    a, b = (make_env(n, limit, obstacles, obs_mode, seed=seed) for _ in range(2))
    _, reached, st = fragments_equal_single_steps(a, b, T=T, fragments=fragments,
                                                  generator=torch.Generator(device="cuda").manual_seed(seed + 1))
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
    _, _, reached = k1_fragments_vs_c_oracle(env, seed, T=T, fragments=3)
    assert reached >= n * 3 * T // 20, reached
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
    act = uniform_actions(a, torch.Generator(device="cuda").manual_seed(7), 2 * T)
    obs_a, rew_a, flg_a = fragment_buffers(2 * T, n)
    obs_b, rew_b, flg_b = fragment_buffers(2 * T, n)
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
