"""Shared set-up and checks of the GPU test modules: the parity bars and observation checks, env factories for the
workloads that recur, the oracle that matches an env's configuration, the dynamic-mode lock step, and the two fragment
checks (fragments against single steps, K1 fragments against the C oracle).  Imported by GPU modules only, after their
pytest.importorskip("torch")."""
import numpy as np
import torch

from oracle.c_dyn_oracle import CDynOracleBatch, DynEnvConfig
from oracle.c_oracle import COracleBatch
from oracle.reach_oracle import OracleBatch, OracleChain, OracleConfig
from pioneer_b200 import BatchConfig, BatchedPioneerEnv, PioneerKinematicConfig, SimulationConfig, demo_obstacles

# ---------------------------------------------------------------------------------------------
# bars of the kinematic mode (test_gpu_parity.py's header) and the observation check
# ---------------------------------------------------------------------------------------------
POS_TOL = 2e-4
REW_TOL = 1e-3
TRIG_TOL = 5e-7

# observation columns (pioneer_knm_env.py:194-211): value blocks and their cos / sin blocks
VALUE_COLS = np.r_[0:6, 18:24, 36:42, 54:60, 72:78, 90:96, 108:114, 129:132]
TRIG_COLS = np.r_[6:18, 24:36, 42:54, 60:72, 78:90, 96:108, 114:126]
POS_COLS = np.r_[126:129, 132:136]


def check_obs(obs_gpu, obs_ref, what=""):
    obs_gpu = np.asarray(obs_gpu, np.float64)
    obs_ref = np.asarray(obs_ref, np.float64)
    assert np.array_equal(obs_gpu[..., VALUE_COLS], obs_ref[..., VALUE_COLS].astype(np.float32)), what
    np.testing.assert_allclose(obs_gpu[..., TRIG_COLS], obs_ref[..., TRIG_COLS], rtol=0, atol=TRIG_TOL, err_msg=what)
    np.testing.assert_allclose(obs_gpu[..., POS_COLS], obs_ref[..., POS_COLS], rtol=0, atol=POS_TOL, err_msg=what)
    np.testing.assert_allclose(obs_gpu[..., 136], obs_ref[..., 136], rtol=0, atol=REW_TOL, err_msg=what)


# ---------------------------------------------------------------------------------------------
# envs
# ---------------------------------------------------------------------------------------------
PENALTY = 0.5
PD = dict(gravity=9.81, kp=2000.0, kd=500.0, torque_scale=1e5)          # bench.py's dynamic-mode workload
BULLET = dict(link_damping=0.04, max_velocity=100.0, motor_kp=0.1, motor_kd=1.0, motor_max_force=5e4)
BULLET_BARS = (5e-5, 5e-6, 2e-3, 2e-4)          # lockstep bars of Bullet-like stepping: the motor solve divides by dt
CONTROL = {"pd": PD, "bullet": dict(gravity=9.81, stepping="bullet", **BULLET), "torque": {}}


def _obstacle_fields():
    return dict(obstacles=demo_obstacles(), contact_penalty=PENALTY, random_box=True)


def kinematic_env(n, *, obstacles=False, seed=0, env_id_base=0, **fields):
    """A kinematic BatchedPioneerEnv.  obstacles=True: the demo obstacles, contact penalty 0.5 and a box redrawn at every
    reset.  Other fields go to PioneerKinematicConfig where it has them, to BatchConfig otherwise, and override the
    obstacle bundle."""
    fields = {**(_obstacle_fields() if obstacles else {}), **fields}
    pc = {k: fields.pop(k) for k in list(fields) if k in PioneerKinematicConfig.__dataclass_fields__}
    return BatchedPioneerEnv(n, seed=seed, env_id_base=env_id_base, pioneer_config=PioneerKinematicConfig(**pc),
                             batch_config=BatchConfig(**fields))


def dynamic_env(n, *, control="pd", obstacles=False, seed=0, env_id_base=0, **fields):
    """A dynamic-mode BatchedPioneerEnv.  control: "pd" (PD position control under gravity), "bullet" (Bullet-like motors
    under gravity) or "torque" (the actions are joint torques; pass gravity and torque_scale).  obstacles=True as in
    kinematic_env.  Other fields: gravity goes to SimulationConfig, the rest to BatchConfig, overriding the bundles."""
    fields = {**CONTROL[control], **(_obstacle_fields() if obstacles else {}), **fields}
    gravity = fields.pop("gravity", 0.0)
    return BatchedPioneerEnv(n, seed=seed, env_id_base=env_id_base, simulation_config=SimulationConfig(gravity=gravity),
                             batch_config=BatchConfig(mode="dynamic", **fields))


def host_boxes(env):
    return env.boxes().cpu().numpy().astype(np.float64)


# ---------------------------------------------------------------------------------------------
# the oracle configured like an env
# ---------------------------------------------------------------------------------------------
def _oracle_fields(env):
    """The settings the kinematic and the dynamic oracle configurations share, read from the env."""
    pc, sc, bc = env.config, env.simulation_config, env.batch_config
    return dict(done_distance=pc.done_distance, award_max=pc.award_max, award_done=pc.award_done,
                award_potential_slope=pc.award_potential_slope, penalty_step=pc.penalty_step, target_lo=pc.target_lo,
                target_hi=pc.target_hi, timestep=sc.timestep, frame_skip=sc.frame_skip,
                max_episode_steps=bc.max_episode_steps, contact_penalty=bc.contact_penalty,
                obstacles=tuple((o.kind, o.position, o.extent) for o in bc.obstacles),
                random_box=(bc.box_pos_lo, bc.box_pos_hi, bc.box_size_lo, bc.box_size_hi) if bc.random_box else None)


def c_oracle_for(env, seed, *, compiled=True):
    """The kinematic oracle of a kinematic env: the C restatement (oracle/reach_oracle.c), or with compiled=False the
    Python one (oracle/reach_oracle.py)."""
    pc, bc = env.config, env.batch_config
    cfg = OracleConfig(max_v_to_r=pc.max_v_to_r, max_a_to_v=pc.max_a_to_v, **_oracle_fields(env))
    batch = COracleBatch if compiled else OracleBatch
    return batch(OracleChain.from_model(env.chain), env.n_envs, cfg, arith={"f32": "np2", "legacy64": "legacy"}[bc.arith],
                 env_id_base=env.env_id_base, seed=seed, auto_reset=bc.auto_reset, obs_mode=bc.obs_mode)


def c_dyn_oracle_for(env, seed):
    """The float64 oracle of a dynamic-mode env (oracle/dynamics_oracle.c)."""
    bc = env.batch_config
    cfg = DynEnvConfig(gravity=env.simulation_config.gravity, kp=bc.kp, kd=bc.kd, torque_scale=bc.torque_scale,
                       stepping=bc.stepping, link_damping=bc.link_damping, max_velocity=bc.max_velocity,
                       motor_kp=bc.motor_kp, motor_kd=bc.motor_kd, motor_max_force=bc.motor_max_force, **_oracle_fields(env))
    return CDynOracleBatch(env.chain, env.n_envs, cfg, env_id_base=env.env_id_base, seed=seed, auto_reset=bc.auto_reset,
                           obs_mode=bc.obs_mode)


# ---------------------------------------------------------------------------------------------
# the dynamic mode in lock step with its oracle (test_gpu_dynamic_parity.py's header)
# ---------------------------------------------------------------------------------------------
def check_dyn_obs(obs, o_obs, worst):
    """obs: device float32 [n,137]; o_obs: oracle float64 computed from the SAME float32 (q, qd, a)."""
    d = np.abs(obs.astype(np.float64) - o_obs)
    for cols in (slice(0, 6), slice(90, 96), slice(108, 114), slice(18, 24), slice(36, 42), slice(129, 132)):
        assert not d[:, cols].any(), f"value columns {cols} must be bit-exact"
    worst["trig"] = max(worst.get("trig", 0.0), float(d[:, 6:90].max()), float(d[:, 96:108].max()), float(d[:, 114:126].max()))
    worst["ptr"] = max(worst.get("ptr", 0.0), float(d[:, 126:129].max()), float(d[:, 132:136].max()))
    worst["pot"] = max(worst.get("pot", 0.0), float(d[:, 136].max()))


def lockstep(env, orc, steps, action_fn, obs_mode="terminal", check_every=1, bars=(5e-6, 5e-7, 5e-5, 5e-6)):
    n = env.n_envs
    s0, o0 = env.state(), orc.state()
    assert np.array_equal(s0["r"].cpu().numpy().astype(np.float64), o0["q"])         # same Philox reset draws
    assert np.array_equal(s0["target"].cpu().numpy().astype(np.float64), o0["target"])
    worst = {}
    n_done = pairs = free_pairs = 0
    for t in range(steps):
        act = action_fn(t)
        obs, reward, flags = env.step_tensor(torch.as_tensor(act).cuda())
        obs, reward, flags = obs.cpu().numpy(), reward.cpu().numpy(), flags.cpu().numpy()
        if obs_mode == "terminal":
            q32, qd32, mask = obs[:, 0:6], obs[:, 90:96], None                        # the post-substep state of EVERY env
        else:                                                                         # finished rows show the next episode
            mask = (flags & 1) == 0
            st = env.state()
            q32, qd32 = st["r"].cpu().numpy(), st["v"].cpu().numpy()
        out = orc.step(act, adopt=(q32, qd32, None if mask is None else mask.astype(np.uint8)), want_obs=(t % check_every == 0))
        # ---- the dynamics: where float64 arrives from the same float32 start.  An inelastic joint stop is a discontinuity
        # (qd := 0): an env in which either side ran into a stop during this step may legitimately differ by qd * dt, so the
        # bars apply to the envs that stayed clear of the stops on both sides; the others are counted
        at_stop = ((q32 <= env.r_lo) | (q32 >= env.r_hi)).any(axis=1)
        free = (out["touched"] == 0) & ~at_stop
        if mask is not None:
            free &= mask
        pairs += int(n if mask is None else mask.sum())
        free_pairs += int(free.sum())
        dq = np.abs(q32.astype(np.float64) - out["own_q"])[free]
        dqd = np.abs(qd32.astype(np.float64) - out["own_qd"])[free]
        if dq.size:
            bar_q = bars[0] + bars[1] * np.abs(out["own_q"][free])
            bar_qd = bars[2] + bars[3] * np.abs(out["own_qd"][free])
            if not (dq <= bar_q).all() or not (dqd <= bar_qd).all():
                i, j = np.unravel_index(np.argmax(dq / bar_q), dq.shape)
                i2, j2 = np.unravel_index(np.argmax(dqd / bar_qd), dqd.shape)
                rows = np.nonzero(free)[0]
                raise AssertionError(f"step {t}: dq {dq[i, j]:.3e} (bar {bar_q[i, j]:.3e}) env {rows[i]} joint {j} qd "
                                     f"{out['own_qd'][rows[i]]}; dqd {dqd[i2, j2]:.3e} (bar {bar_qd[i2, j2]:.3e}) env {rows[i2]} "
                                     f"joint {j2} qd {out['own_qd'][rows[i2]]} q {out['own_q'][rows[i2]]} act {act[rows[i2]]}")
            worst["dq"] = max(worst.get("dq", 0.0), float(dq.max()))
            worst["dqd"] = max(worst.get("dqd", 0.0), float(dqd.max()))
            worst["qd_abs"] = max(worst.get("qd_abs", 0.0), float(np.abs(out["own_qd"][free]).max()))
        # ---- the env layer on identical inputs
        assert np.array_equal(flags, out["flags"]), (t, int((flags != out["flags"]).sum()))
        dr = np.abs(reward.astype(np.float64) - out["reward"])
        if mask is not None:
            dr = dr[mask]                                                             # finished rows: the oracle used its own q
        if dr.size:
            assert dr.max() <= 2e-3, (t, float(dr.max()))
            worst["reward"] = max(worst.get("reward", 0.0), float(dr.max()))
        if out["obs"] is not None:
            check_dyn_obs(obs, out["obs"], worst)
        n_done += int((flags & 1).sum())
    assert worst.get("trig", 0.0) <= 1e-6 and worst.get("ptr", 0.0) <= 2e-4 and worst.get("pot", 0.0) <= 1e-3, worst
    worst["free_fraction"] = free_pairs / max(pairs, 1)
    # ---- after the run: the reset envs carry the oracle's Philox draws, counters and statistics agree
    s, o = env.state(), orc.state()
    assert np.array_equal(s["t"].cpu().numpy(), o["t"])
    assert np.array_equal(s["target"].cpu().numpy().astype(np.float64), o["target"])
    assert np.array_equal(s["r"].cpu().numpy().astype(np.float64), o["q"])            # adopted or freshly reset: identical
    assert np.abs(s["potential"].cpu().numpy() - o["potential"]).max() <= 1e-3
    assert np.abs(s["ep_return"].cpu().numpy() - o["ep_return"]).max() <= 5e-2
    st, os_ = env.episode_stats(), orc.stats
    assert st["episodes"] == os_[0] == n_done and st["sum_length"] == os_[2] and st["env_steps"] == os_[6] == steps * n
    assert st["reached_target"] == os_[7]
    if n_done:
        assert abs(st["sum_return"] - os_[1]) <= 5e-2 * n_done and abs(st["max_return"] - os_[4]) <= 5e-2
        assert abs(st["min_return"] - os_[5]) <= 5e-2
    return worst, n_done


def setpoints(env, seed, hold=25):
    """New PD set points every `hold` steps (uniform in the joint range): long transients, joints driven into the stops."""
    rng = np.random.default_rng(seed)
    cache = {}

    def fn(t):
        k = t // hold
        if k not in cache:
            cache.clear()
            cache[k] = rng.uniform(env.r_lo, env.r_hi, size=(env.n_envs, 6)).astype(np.float32)
        return cache[k]
    return fn


# ---------------------------------------------------------------------------------------------
# fragments (pnr_step_many)
# ---------------------------------------------------------------------------------------------
STATE_KEYS = ("r", "v", "a", "potential", "target", "t", "ep_return")
STAT_KEYS = ("episodes", "sum_length", "env_steps", "reached_target", "max_return", "min_return")


def fragment_buffers(T, n):
    """Zero-filled obs [T, n, 137], reward [T, n] and flags [T, n] of a fragment, with every obs[t] on a 16-byte boundary."""
    n_pad = (n + 3) // 4 * 4
    return (torch.zeros((T, n_pad, 137), device="cuda")[:, :n], torch.zeros((T, n), device="cuda"),
            torch.zeros((T, n), dtype=torch.uint8, device="cuda"))


def uniform_actions(env, generator, T):
    """T steps of actions drawn uniformly from the env's action space on the device: [T, n, 6]."""
    lo, hi = torch.as_tensor(env.action_space.low).cuda(), torch.as_tensor(env.action_space.high).cuda()
    return lo + torch.rand((T, env.n_envs, 6), device="cuda", generator=generator) * (hi - lo)


def reached_resets(flags):
    """Episodes that ended because the target was reached (done, not truncated by the TimeLimit)."""
    f = flags.to(torch.int32)
    return int(((f & 1) != 0).logical_and((f & 2) == 0).sum())


def assert_same_envs(a, b, what):
    sa, sb = a.state(), b.state()
    for key in STATE_KEYS:
        assert torch.equal(sa[key], sb[key]), (what, key)
    if a.batch_config.random_box:                  # only a random-box handle keeps per-env boxes
        assert torch.equal(a.boxes(), b.boxes()), what


def assert_same_stats(a, b, return_rtol=1e-9):
    """Episode counts, lengths and extreme returns exactly.  The return sums to return_rtol: they are float64 atomics,
    added per warp in an order that depends on the launch shape, and the squared returns are rounded products."""
    st_a, st_b = a.episode_stats(), b.episode_stats()
    for key in STAT_KEYS:
        assert st_a[key] == st_b[key], (key, st_a[key], st_b[key])
    for key in ("sum_return", "sum_return_sq"):
        assert abs(st_a[key] - st_b[key]) <= return_rtol * abs(st_b[key]), (key, st_a[key], st_b[key])
    return st_a


def fragments_equal_single_steps(a, b, *, T, fragments, generator, filters=None, return_rtol=1e-9):
    """Twin envs: `a` runs fragments of T steps in one launch, `b` the same actions one step per launch.  Flags, rewards
    and observations agree bit for bit at every step, state and boxes after every fragment, the episode statistics at
    the end (assert_same_stats).  filters: the twins' fused MeanStdObsFilter pair.  A first fragment then runs under the
    identity (nothing synchronised yet); both sides synchronise and are given the same statistics, so that the
    `fragments` compared after it normalise with non-trivial applied statistics, and the statistics agree at the end.
    Returns (resets, `reached` resets, a's episode statistics); closes neither env."""
    n = a.n_envs
    obs, rew, flg = fragment_buffers(T, n)
    n_done = reached = 0

    def fragment(k):
        nonlocal n_done, reached
        act = uniform_actions(a, generator, T)
        a.step_many(act, obs, rew, flg)
        for t in range(T):
            o, r, f = b.step_tensor(act[t])
            assert torch.equal(f, flg[t]), (k, t, int((f != flg[t]).sum()))
            assert torch.equal(r, rew[t]), (k, t, float((r - rew[t]).abs().max()))
            assert torch.equal(o, obs[t]), (k, t, float((o - obs[t]).abs().max()))
        assert_same_envs(a, b, k)
        n_done += int((flg & 1).sum())
        reached += reached_resets(flg)

    def same_filter_statistics():
        fa, fb = filters
        fa.sync(); fb.sync()
        (na, ma, va), (nb, mb, vb) = fa._get(), fb._get()
        assert na == nb                            # float64 atomics in a different order: sums agree to rounding
        np.testing.assert_allclose(ma, mb, rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(va, vb, rtol=1e-9, atol=1e-12)
        return na, ma, va

    if filters:
        fragment(-1)
        stats = same_filter_statistics()
        assert np.abs(stats[1]).max() > 1.0        # the applied statistics are no longer the identity
        for f in filters:
            f.set_stats(*stats)
    for k in range(fragments):
        fragment(k)
    if filters:
        same_filter_statistics()
    assert n_done > 0                              # resets (and box redraws) happened inside the fragments
    return n_done, reached, assert_same_stats(a, b, return_rtol)


def k1_fragments_vs_c_oracle(env, seed, *, T, fragments):
    """A kinematic env runs `fragments` fragments of T steps beside the C oracle of the same seed, both fed actions drawn
    with numpy's generator of that seed.  Flags exactly and rewards within 2e-3 at every step; after every fragment the
    last step's observation (check_obs), r, v, a, t and target exactly, and the boxes of a random-box env; at the end
    episodes, sum_length and reached_target.  Returns (worst reward deviation, resets, `reached` resets)."""
    n = env.n_envs
    orc = c_oracle_for(env, seed)
    rng = np.random.default_rng(seed)
    obs, rew, flg = fragment_buffers(T, n)
    worst, n_done, reached = 0.0, 0, 0
    for k in range(fragments):
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
        if env.batch_config.random_box:
            assert np.array_equal(host_boxes(env), orc.boxes()), k
        n_done += int((flg_h & 1).sum())
        reached += reached_resets(flg)
    assert worst <= 2e-3, worst
    st = env.episode_stats()
    assert st["episodes"] == orc.stats[0] == n_done, (st["episodes"], orc.stats[0], n_done)
    assert st["sum_length"] == orc.stats[2] and st["reached_target"] == orc.stats[7]
    return worst, n_done, reached
