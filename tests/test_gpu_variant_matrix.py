"""Every step-kernel variant the library can launch, in both launch shapes, against the oracles.

pnr_launch_step picks one of ten K1 instantiations pnr_step_kernel<ARITH, OBS_MODE, OBSTACLES, FILTER>; K2
(pnr_dynamic_kernel.cuh) is templated on <OBS_MODE, OBSTACLES, CHAIN, STEPPING> with a run-time filter switch.  Each runs
as one step per launch (pnr_step) or as a fragment of T steps in one launch (pnr_step_many).  The other GPU modules cover
the plain corners of this matrix; this one covers the rest:

  1. K1 single step with obstacles + a per-env random box in the arithmetic / observation modes test_gpu_obstacles.py does
     not run, against the C oracle (oracle/reach_oracle.c): state, flags and boxes bit-exact, reward within 2e-3.
  2. Fragments equal single steps bit for bit for every combination pnr_step_many can launch (K1 and K2, obstacles, random
     box, fused filter, both observation modes, both K2 steppings), ragged sizes and several tiles per CTA / warp.
  3. The bench's kinematic obstacle workload (16,384 envs, random box, fragments of 8) straight against the C oracle.
  4. K2 lock step (oracle/dynamics_oracle.c) for obstacles x auto-reset observations and Bullet-like stepping x obstacles.
  5. The fused normaliser's statistics at 1M rows (K1) / 131,072 rows (K2) against float64 column sums of the raw rows.
  6. RolloutWorker's normalised observations (fused filter + pnr_observe_done) against oracle/filter_oracle.py."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle.filter_oracle import BatchSyncFilter
from tests._gpu import (BULLET_BARS, c_dyn_oracle_for, c_oracle_for, check_obs, dynamic_env, fragment_buffers,
                        fragments_equal_single_steps, host_boxes, k1_fragments_vs_c_oracle, kinematic_env, lockstep,
                        setpoints, uniform_actions)

pytestmark = pytest.mark.gpu


# ---------------------------------------------------------------------------------------------
# 1. K1 single step with obstacles + random box in the modes test_gpu_obstacles.py does not run
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [77, 4096 + 37])
@pytest.mark.parametrize("arith,obs_mode", [("legacy64", "terminal"), ("f32", "autoreset"), ("legacy64", "autoreset")])
def test_kinematic_obstacles_single_step_vs_c_oracle(arith, obs_mode, n):
    """TimeLimit 7 over 24 steps: three auto-resets per env, each redrawing the env's box; 77 envs = two full warp tiles and
    a ragged one.  In auto-reset observation mode a finished row shows the oracle's fresh episode."""
    seed, steps = 31, 24
    env = kinematic_env(n, arith=arith, obs_mode=obs_mode, max_episode_steps=7, obstacles=True, seed=seed)
    orc = c_oracle_for(env, seed)
    assert np.array_equal(host_boxes(env), orc.boxes())
    rng = np.random.default_rng(seed)
    worst_rew, n_done = 0.0, 0
    for t in range(steps):
        act = (rng.uniform(-1, 1, size=(n, 6)) * env.a_max).astype(np.float32)
        obs, reward, flags = env.step_tensor(torch.as_tensor(act).cuda())
        o_obs, o_rew, o_flags = orc.step(act)
        f = flags.cpu().numpy()
        assert np.array_equal(f, o_flags), f"flags differ at step {t}"
        s, o = env.state(), orc.state()
        for k in ("r", "v", "a", "t"):
            assert np.array_equal(s[k].cpu().numpy(), o[k]), (k, t)
        assert np.array_equal(s["target"].cpu().numpy(), o["target"].astype(np.float32)), t
        assert np.abs(s["ep_return"].cpu().numpy() - o["ep_return"]).max() <= 2e-3 * 7, t
        assert np.array_equal(host_boxes(env), orc.boxes()), f"boxes differ after step {t}"
        worst_rew = max(worst_rew, float(np.abs(reward.cpu().numpy() - o_rew).max()))
        ob = obs.cpu().numpy()
        check_obs(ob, o_obs, f"step {t}")
        done = (f & 1) != 0
        if obs_mode == "autoreset" and done.any():        # the first observation of the new episode, not the terminal one
            assert (o["t"][done] == 0).all()
            assert np.array_equal(ob[done, 0:6], o["r"][done])
            assert np.array_equal(ob[done, 129:132], o["target"][done].astype(np.float32))
            assert (ob[done, 90:96] == 0).all() and (ob[done, 108:114] == 0).all()
        n_done += int(done.sum())
    assert worst_rew <= 2e-3, worst_rew
    assert n_done >= 3 * n
    st = env.episode_stats()
    assert st["episodes"] == orc.stats[0] == n_done and st["env_steps"] == orc.stats[6] == n * steps
    assert st["sum_length"] == orc.stats[2] and st["reached_target"] == orc.stats[7]
    print(f"K1 {arith}/{obs_mode}/obstacles+random box, {n} envs: worst reward deviation {worst_rew:.3e}")
    env.close()


# ---------------------------------------------------------------------------------------------
# 2. fragments (pnr_step_many) equal single steps (pnr_step), bit for bit, for every combination
# ---------------------------------------------------------------------------------------------
def twins_equal(make, fused, seed):
    """Fragments of 8 against single steps on twin envs (three fragments, after a first one under the identity filter
    when the fused filter is on)."""
    from pioneer_b200.obs_filter import MeanStdObsFilter
    a, b = make(), make()
    filters = (MeanStdObsFilter(a, fused=True), MeanStdObsFilter(b, fused=True)) if fused else None
    fragments_equal_single_steps(a, b, T=8, fragments=3, generator=torch.Generator(device="cuda").manual_seed(seed),
                                 filters=filters)
    a.close(); b.close()


SMALL, KIN_LARGE, DYN_LARGE = 4096 + 37, 300000 + 17, 131072 + 5
KIN_CASES = [(arith, obs_mode, obstacles, False, SMALL) for arith in ("f32", "legacy64")
             for obs_mode in ("terminal", "autoreset") for obstacles in (False, True)] \
    + [("f32", "terminal", obstacles, True, SMALL) for obstacles in (False, True)] \
    + [("f32", "terminal", True, False, KIN_LARGE), ("legacy64", "autoreset", True, False, KIN_LARGE),
       ("f32", "terminal", True, True, KIN_LARGE)]


@pytest.mark.parametrize("arith,obs_mode,obstacles,fused,n", KIN_CASES)
def test_kinematic_fragment_equals_single_steps(arith, obs_mode, obstacles, fused, n):
    """K1 (the fused filter exists for float32 terminal observations only; the API refuses the rest).  TimeLimit 4 with
    fragments of 8: every env resets twice inside each fragment."""
    twins_equal(lambda: kinematic_env(n, arith=arith, obs_mode=obs_mode, max_episode_steps=4, obstacles=obstacles, seed=6),
                fused, seed=1)


DYN_CASES = [(obs_mode, obstacles, stepping, False, SMALL) for obs_mode in ("terminal", "autoreset")
             for obstacles in (False, True) for stepping in ("explicit", "bullet")] \
    + [("terminal", False, "explicit", True, SMALL), ("autoreset", True, "explicit", True, SMALL),
       ("terminal", True, "bullet", True, SMALL)] \
    + [("terminal", True, "explicit", False, DYN_LARGE), ("autoreset", True, "bullet", False, DYN_LARGE),
       ("terminal", True, "explicit", True, DYN_LARGE)]


@pytest.mark.parametrize("obs_mode,obstacles,stepping,fused,n", DYN_CASES)
def test_dynamic_fragment_equals_single_steps(obs_mode, obstacles, stepping, fused, n):
    """K2: the warp keeps its tile's env state in registers across the fragment; TimeLimit 5 with fragments of 8."""
    control = "pd" if stepping == "explicit" else stepping
    twins_equal(lambda: dynamic_env(n, control=control, obs_mode=obs_mode, max_episode_steps=5, obstacles=obstacles, seed=8),
                fused, seed=2)


# ---------------------------------------------------------------------------------------------
# 3. bench.py's kinematic obstacle workload, fragments of 8, against the C oracle
# ---------------------------------------------------------------------------------------------
def test_kinematic_obstacle_fragments_vs_c_oracle():
    """16,384 envs, random box, TimeLimit 25, eight fragments of 8 through pnr_step_many; the oracle steps eight times per
    fragment.  Flags and reward every step; r, v, boxes and the observation at the end of every fragment."""
    n, T, seed = 16384, 8, 44
    env = kinematic_env(n, max_episode_steps=25, obstacles=True, seed=seed)
    worst, n_done, _ = k1_fragments_vs_c_oracle(env, seed, T=T, fragments=8)
    assert n_done >= 2 * n
    print(f"K1 obstacle fragments vs C oracle, {n} envs x {8 * T} steps: worst reward deviation {worst:.3e}")
    env.close()


# ---------------------------------------------------------------------------------------------
# 4. K2 lock step for the single-step instantiations test_gpu_dynamic_parity.py does not run
# ---------------------------------------------------------------------------------------------
def test_dynamic_obstacles_random_box_autoreset_lockstep():
    n = 4096
    env = dynamic_env(n, obs_mode="autoreset", max_episode_steps=20, obstacles=True, seed=23)
    orc = c_dyn_oracle_for(env, 23)
    assert np.array_equal(host_boxes(env), orc.state()["box"])
    worst, n_done = lockstep(env, orc, 45, setpoints(env, 11), obs_mode="autoreset", check_every=5)
    assert n_done >= 2 * n and worst["free_fraction"] > 0.85, (n_done, worst)
    assert np.array_equal(host_boxes(env), orc.state()["box"])      # redrawn twice, same draws
    print("K2 obstacles + random box, autoreset observations, worst:", worst)
    env.close()


def test_dynamic_bullet_stepping_with_obstacles_lockstep():
    n = 4096
    env = dynamic_env(n, control="bullet", max_episode_steps=25, obstacles=True, seed=15)
    orc = c_dyn_oracle_for(env, 15)
    assert np.array_equal(host_boxes(env), orc.state()["box"])
    worst, n_done = lockstep(env, orc, 60, setpoints(env, 12, hold=12), check_every=4, bars=BULLET_BARS)
    assert n_done >= 2 * n and worst["free_fraction"] > 0.5, (n_done, worst)
    assert np.array_equal(host_boxes(env), orc.state()["box"])
    print("K2 Bullet-like stepping + obstacles + random box, worst:", worst)
    env.close()


# ---------------------------------------------------------------------------------------------
# 5. the fused normaliser's statistics at scale against float64
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["kinematic", "dynamic"])
def test_fused_filter_statistics_at_scale_vs_float64(mode):
    """1,048,576 envs (K1) / 131,072 envs (K2), fragments of 8, MeanStdObsFilter(fused=True).  An unfused twin driven by
    the same actions supplies the raw rows; the truth is their column mean and unbiased variance in float64 (sums about a
    fixed shift near the mean, one step of rows at a time on the device).  Checked after the first sync (the fragment ran
    under the identity, so K1's task warp accumulated the raw tail columns, e.g. target x in [15, 25], in its float32
    per-lane partials) and after the second."""
    from pioneer_b200.obs_filter import MeanStdObsFilter
    n, T = (1 << 20, 8) if mode == "kinematic" else (131072, 8)
    make = kinematic_env if mode == "kinematic" else dynamic_env
    a, b = make(n, max_episode_steps=6, seed=3), make(n, max_episode_steps=6, seed=3)
    fa = MeanStdObsFilter(a, fused=True)
    g = torch.Generator(device="cuda").manual_seed(4)
    (obs_a, rew_a, flg_a), (obs_b, rew_b, flg_b) = fragment_buffers(T, n), fragment_buffers(T, n)
    shift, s1, s2, rows = None, None, None, 0
    report = []
    for it in range(2):
        act = uniform_actions(a, g, T)
        a.step_many(act, obs_a, rew_a, flg_a)
        b.step_many(act, obs_b, rew_b, flg_b)
        assert torch.equal(flg_a, flg_b) and torch.equal(rew_a, rew_b)
        for t in range(T):
            x = obs_b[t].double()
            if shift is None:
                shift = x[:4096].mean(0)
                s1, s2 = torch.zeros_like(shift), torch.zeros_like(shift)
            d = x - shift
            s1 += d.sum(0)
            s2 += (d * d).sum(0)
            del x, d
        rows += T * n
        fa.sync()
        mean_true = (shift + s1 / rows).cpu().numpy()
        var_true = ((s2 - s1 * s1 / rows) / (rows - 1)).cpu().numpy()
        f_n, f_mean, f_var = fa._get()
        assert f_n == rows, (f_n, rows)
        err_mean = np.abs(f_mean - mean_true) - 1e-6 * np.abs(mean_true)
        assert (err_mean <= 1e-6).all(), (it, int(np.argmax(err_mean)), float(err_mean.max()))
        moving = var_true > 0
        rel = np.abs(f_var[moving] - var_true[moving]) / var_true[moving]
        worst_col = int(np.nonzero(moving)[0][np.argmax(rel)])
        report.append(f"sync {it + 1}: worst relative variance error {rel.max():.3e} (column {worst_col}), "
                      f"tail columns 126-136 {rel[np.nonzero(moving)[0] >= 126].max():.3e}")
        assert (np.abs(f_var[~moving]) <= 1e-12).all(), f_var[~moving]        # constant columns
        assert rel.max() <= 1e-5, report[-1]
    print(f"fused filter statistics, {mode}, {n} envs x {T} steps per sync: " + "; ".join(report))
    a.close(); b.close()


# ---------------------------------------------------------------------------------------------
# 6. RolloutWorker's normalised observations, not just their bounds
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cuda_graph", [False, True])
def test_rollout_worker_fused_filter_values_vs_the_filter_oracle(cuda_graph):
    """Eager or graph-replayed RolloutWorker with the fused filter (its default): terminal observations, in-kernel auto-reset,
    pnr_observe_done rewriting finished rows, 512 + 3 envs (a ragged last tile), T = 6, TimeLimit 4, four collect() + sync()
    rounds.  An unfused twin replays the worker's recorded actions (from a graph of its own when the worker replays one);
    BatchSyncFilter sees the rows the device pushed, in the same order (reset rows, every step's rows, then the fresh rows of
    the finished envs) and synchronises at the same points."""
    from pioneer_b200 import BatchConfig, BatchedPioneerEnv
    from pioneer_b200.rollout import RolloutWorker
    n, T, rounds = 512 + 3, 6, 4
    make = lambda: BatchedPioneerEnv(n, seed=13, batch_config=BatchConfig(max_episode_steps=4))   # noqa: E731
    env, twin = make(), make()
    w = RolloutWorker(env, fragment_length=T, seed=3, cuda_graph=cuda_graph)
    assert w.fused
    warm = []
    if cuda_graph:
        # the first collect() runs the T steps once eagerly before it captures them; record those actions too
        run_steps = w._steps

        def recording_steps():
            run_steps()
            if not torch.cuda.is_current_stream_capturing():
                warm.append(w.actions.clone())
        w._steps = recording_steps
    ora = BatchSyncFilter(137)
    act_buf = torch.empty((T, n, 6), device="cuda")
    raw, rew, flg = fragment_buffers(T, n)
    rows = fragment_buffers(T, n)[0]

    def twin_steps(k):
        for t in range(k):
            twin.step_tensor(act_buf[t], out=(raw[t], rew[t], flg[t]))
            rows[t].copy_(raw[t])
            twin.observe_done(flg[t], rows[t])         # finished rows: the first observation of the next episode

    def oracle_rows(k):
        """The normalised rows the worker must have produced in the twin's last k steps (pushed in the device's order)."""
        wants, done_total = [], 0
        for t in range(k):
            ora(raw[t].cpu().numpy())                  # the step kernel pushes every row it writes
            r, done = rows[t].cpu().numpy(), (flg[t].cpu().numpy() & 1) != 0
            if done.any():
                ora(r[done])                           # pnr_observe_done pushes the rows it rewrites
            wants.append(ora(r, update=False))
            done_total += int(done.sum())
        return wants, done_total

    reset_rows = twin.reset().cpu().numpy()
    ora(reset_rows)
    ora.sync()
    prev = ora(reset_rows, update=False)
    twin_graph = None
    worst, n_done = 0.0, 0
    for it in range(rounds):
        out = w.collect()
        if it == 0 and cuda_graph:
            assert len(warm) == 1
            act_buf.copy_(warm[0])
            twin_steps(T)
            prev = oracle_rows(T)[0][-1]
            # steps captured in a graph draw their resets from the graph's own key domain, keyed by the ticks frozen at
            # capture plus the device-side advance of every replay: the twin's steps are captured and replayed the same way
            torch.cuda.synchronize()
            twin_graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(twin_graph):
                twin.advance_reset_counter(T)
                twin_steps(T)
        act_buf.copy_(out["actions"])
        if twin_graph is not None:
            twin_graph.replay()
        else:
            twin_steps(T)
        wants, k = oracle_rows(T)
        n_done += k
        got = out["obs"].cpu().numpy()
        assert np.abs(got[0] - prev).max() <= 2e-5, (it, float(np.abs(got[0] - prev).max()))
        nxt = out["next_obs"].cpu().numpy()
        for t in range(T):
            d = float(np.abs(nxt[t] - wants[t]).max())
            worst = max(worst, d)
            assert d <= 2e-5, (it, t, d, np.unravel_index(np.argmax(np.abs(nxt[t] - wants[t])), wants[t].shape))
        prev = wants[-1]
        w.sync()
        ora.sync()
        f_n, f_mean, f_var = w.filter._get()
        assert f_n == ora.rs.n, (it, f_n, ora.rs.n)
        np.testing.assert_allclose(f_mean, ora.rs.M, rtol=1e-6, atol=1e-6)
        np.testing.assert_allclose(f_var, ora.rs.var, rtol=1e-5, atol=1e-9)
    assert n_done >= rounds * T * n // 4 - n
    print(f"RolloutWorker (cuda_graph={cuda_graph}): worst normalised-observation deviation {worst:.3e}, {n_done} resets")
    env.close(); twin.close()
