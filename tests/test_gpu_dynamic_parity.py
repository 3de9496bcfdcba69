"""Dynamic (Tier-B) mode on the GPU against the compiled float64 oracle (oracle/dynamics_oracle.c) at BASELINE.json's
full sizes: configs[2] = 65,536 envs with joint limits, PD position control, TimeLimit and auto-reset; configs[3] = 16,384
envs with the demo obstacles.  PARITY UNPINNED vs PyBullet (the reference never runs Bullet's dynamics with non-zero
inputs; see the oracle's header) -- the oracle is the float64 definition of this mode, checked on the CPU against the
6x6-matrix Python oracle, CRBA + RNEA and Lagrange's equations.

Method (lock step, see oracle/dynamics_oracle.c): every step the oracle advances from the float32 state the device held
before the step, reports where its own float64 substeps arrive (compared with the device inside the bars below), then
ADOPTS the device's float32 post-step state, so that the env layer -- reward, done / TimeLimit flags, observation,
statistics, Philox auto-reset -- is compared on identical inputs: flags BIT-EXACT, like the kinematic mode.

Bars per env step (10 substeps, float32 vs float64) for every env that stayed clear of the joint stops on both sides during
the step: |dq| <= 5e-6 + 5e-7 |q|,  |dqd| <= 5e-5 + 5e-6 |qd|  (measured on B200 at 65,536 envs x 200 steps: 1.1e-6 and 2.0e-5
with |qd| up to 26 rad/s).  An inelastic stop is a discontinuity (qd := 0): an env in which either side ran into one may
differ by qd * dt in that step, so those (env, step) pairs -- 8 % under PD control with random set points -- are checked
through the env layer only and their share is asserted.
Observation: value columns r, v, a, r_lo, r_hi, target bit-exact; cos / sin columns <= 1e-6; pointer xyz / distance <= 2e-4;
potential <= 1e-3; reward <= 2e-3; episode statistics: counts exact, sums to float32 accumulation."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from tests._gpu import BULLET_BARS, c_dyn_oracle_for, dynamic_env, host_boxes, lockstep, setpoints

pytestmark = pytest.mark.gpu


def test_config3_65536_envs_pd_control_timelimit_autoreset():
    """BASELINE.json configs[2]: 65,536 envs, joint limits, PD position control, TimeLimit + in-kernel auto-reset; 200 steps
    with TimeLimit 64 => every env goes through three episode ends and Philox resets."""
    env = dynamic_env(65536, max_episode_steps=64, seed=12)
    orc = c_dyn_oracle_for(env, 12)
    worst, n_done = lockstep(env, orc, 200, setpoints(env, 1), check_every=10)
    assert n_done >= 3 * 65536 and worst["free_fraction"] > 0.85
    print("config3 dynamic parity, worst:", worst)
    env.close()


def test_autoreset_observation_mode_at_16384_envs():
    env = dynamic_env(16384, obs_mode="autoreset", max_episode_steps=40, seed=5, env_id_base=1 << 33)
    orc = c_dyn_oracle_for(env, 5)
    worst, n_done = lockstep(env, orc, 100, setpoints(env, 2), obs_mode="autoreset", check_every=5)
    assert n_done >= 2 * 16384 and worst["free_fraction"] > 0.85   # (+ the rare env that reaches its target)
    print("autoreset mode, worst:", worst)
    env.close()


def test_torque_control_with_gravity():
    n = 8192
    env = dynamic_env(n, control="torque", gravity=9.81, torque_scale=40.0, max_episode_steps=30, seed=3)
    orc = c_dyn_oracle_for(env, 3)
    rng = np.random.default_rng(4)
    tau_max = (np.asarray(env.chain.effort) * 40.0).astype(np.float32)
    assert np.array_equal(env.action_space.high, tau_max)                            # the action space of this mode
    worst, _ = lockstep(env, orc, 60, lambda t: (rng.uniform(-1.2, 1.2, size=(n, 6)) * tau_max).astype(np.float32))
    print("torque control, worst:", worst)
    assert worst["free_fraction"] > 0.05          # under gravity most arms end up resting on a stop; the rest is compared
    env.close()


def test_config4_16384_envs_with_the_demo_obstacles():
    """BASELINE.json configs[3]: ground plane, the reference demo's box, a sphere; contact penalty in the reward."""
    env = dynamic_env(16384, obstacles=True, random_box=False, max_episode_steps=50, seed=9)
    orc = c_dyn_oracle_for(env, 9)
    worst, n_done = lockstep(env, orc, 100, setpoints(env, 3), check_every=5)
    assert n_done >= 2 * 16384 and worst["free_fraction"] > 0.85
    print("config4 dynamic parity, worst:", worst)
    env.close()


def test_per_env_random_box_in_dynamic_mode():
    n = 4096
    env = dynamic_env(n, obstacles=True, max_episode_steps=20, seed=21)
    orc = c_dyn_oracle_for(env, 21)
    assert np.array_equal(host_boxes(env), orc.state()["box"])
    worst, n_done = lockstep(env, orc, 45, setpoints(env, 5), check_every=5)
    assert n_done >= 2 * n
    assert np.array_equal(host_boxes(env), orc.state()["box"])      # redrawn twice, same draws
    env.close()


def test_bullet_like_stepping_against_the_compiled_oracle():
    """PNR_STEPPING_BULLET (opt-in; restated from memory of btMultiBody, UNPINNED vs PyBullet): per-link damping, POSITION_CONTROL
    motors as velocity-level constraints with impulse clamp, +-100 rad/s clamp -- the device against the float64 restatement
    (oracle/dynamics_oracle.c, stepping = 1), 4,096 envs x 60 steps with gravity, TimeLimit 25 and auto-reset.  The motor solve
    divides by dt, so qd carries 240 x the float32 rounding of q: bars |dq| <= 5e-5 + 5e-6 |q|, |dqd| <= 2e-3 + 2e-4 |qd|."""
    n = 4096
    env = dynamic_env(n, control="bullet", max_episode_steps=25, seed=14)
    orc = c_dyn_oracle_for(env, 14)
    assert np.array_equal(env.action_space.low, env.r_lo)                  # motor set points
    worst, n_done = lockstep(env, orc, 60, setpoints(env, 9, hold=12), check_every=4, bars=BULLET_BARS)
    assert n_done >= 2 * n and worst["free_fraction"] > 0.5
    print("bullet-like stepping, worst:", worst)
    env.close()


def test_free_running_drift_is_bounded_under_pd_control():
    """No adoption: the float64 oracle free-runs beside 8,192 envs for 300 steps (TimeLimit 100, auto-reset).  PD control
    contracts, so the float32 trajectory stays near the float64 one: 99.9 % of the envs within 2e-3 rad at every check, every
    env within 0.25 (an inelastic joint stop is a discontinuity: when one side touches it a substep earlier than the other
    the two differ by up to qd * dt -- 26 rad/s x 1/240 s = 0.11 rad -- until the controller pulls them together again); flags may only differ where the
    distance sits within that drift of the done threshold (never, for random targets)."""
    n = 8192
    env = dynamic_env(n, max_episode_steps=100, seed=31)
    orc = c_dyn_oracle_for(env, 31)
    fn = setpoints(env, 7, hold=50)
    worst, worst_q999 = 0.0, 0.0
    for t in range(300):
        act = fn(t)
        obs, reward, flags = env.step_tensor(torch.as_tensor(act).cuda())
        out = orc.step(act, want_obs=False)
        f = flags.cpu().numpy()
        diff = f != out["flags"]
        assert not diff.any(), (t, int(diff.sum()))
        if t % 10 == 9:
            q = obs[:, 0:6].cpu().numpy().astype(np.float64)
            err = np.abs(q - out["own_q"]).max(axis=1)
            worst = max(worst, float(err.max()))
            worst_q999 = max(worst_q999, float(np.quantile(err, 0.999)))
    print("free-running drift: worst", worst, "99.9 % quantile", worst_q999)
    assert worst <= 0.25 and worst_q999 <= 2e-3, (worst, worst_q999)
    env.close()
