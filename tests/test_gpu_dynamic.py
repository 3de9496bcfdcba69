"""Dynamic (Tier-B) mode on the GPU against the float64 oracle (oracle/dynamics_oracle.py).

PARITY UNPINNED vs PyBullet (the reference never runs Bullet's dynamics with non-zero inputs; see the oracle's
header).  Bars: one env step (10 ABA substeps, float32) from identical float32 states: |dq| <= 2e-5 rad,
|dqd| <= 2e-4 rad/s; free-running 1,000 steps under PD control (a contracting system): |dq| <= 2e-3; the
reference-pinned fact -- zero velocity, gravity and torque leave the state bit-unchanged -- holds exactly."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle.dynamics_oracle import DynChain, DynConfig, dynamic_substeps
from oracle.reach_oracle import OracleChain, fk_pointer

pytestmark = pytest.mark.gpu


def make(n, gravity=0.0, kp=0.0, kd=0.0, torque_scale=1.0, **kw):
    from pioneer_b200 import BatchConfig, BatchedPioneerEnv, SimulationConfig
    bc = BatchConfig(mode="dynamic", kp=kp, kd=kd, torque_scale=torque_scale,
                     max_episode_steps=kw.pop("max_episode_steps", 0), auto_reset=kw.pop("auto_reset", False))
    return BatchedPioneerEnv(n, batch_config=bc, simulation_config=SimulationConfig(gravity=gravity), **kw)


def chain_of(env):
    return DynChain.from_model(env.chain), OracleChain.from_model(env.chain)


def test_zero_input_is_a_bitwise_no_op():
    """SURVEY 8(c) C6 (viii): what World.step() does in the reference (g = 0, qd = 0, tau = 0)."""
    env = make(1000, seed=3)
    before = env.state()
    zero = torch.zeros((1000, 6), device="cuda")
    for _ in range(24):                                    # 240 substeps
        obs, reward, flags = env.step_tensor(zero)
    after = env.state()
    assert torch.equal(after["r"], before["r"]) and torch.equal(after["v"], before["v"])
    assert (after["v"] == 0).all() and (after["t"] == 24).all()
    env.close()


@pytest.mark.parametrize("gravity,kp,kd,scale", [(0.0, 0.0, 0.0, 1.0), (9.81, 0.0, 0.0, 50.0), (9.81, 800.0, 200.0, 1e4),
                                                 (0.0, 300.0, 60.0, 200.0)])
def test_one_step_against_the_float64_oracle(gravity, kp, kd, scale):
    n = 512
    env = make(n, gravity=gravity, kp=kp, kd=kd, torque_scale=scale, seed=11)
    dyn, kin = chain_of(env)
    cfg = DynConfig(gravity=gravity, kp=kp, kd=kd, torque_scale=scale)
    rng = np.random.default_rng(5)
    q0 = rng.uniform(env.r_lo * 0.9, env.r_hi * 0.9).astype(np.float32) * np.ones((n, 1), np.float32)
    q0 = (q0 * rng.uniform(0.2, 1.0, size=(n, 6))).astype(np.float32)
    qd0 = rng.normal(size=(n, 6)).astype(np.float32) * 0.5
    env.set_state(r=q0, v=qd0)
    if kp or kd:
        act = rng.uniform(env.r_lo, env.r_hi, size=(n, 6)).astype(np.float32)       # desired joint positions
    else:
        act = (rng.normal(size=(n, 6)) * scale).astype(np.float32)                  # joint torques
    obs, reward, flags = env.step_tensor(torch.as_tensor(act).cuda())
    s = env.state()
    q1, qd1 = s["r"].cpu().numpy(), s["v"].cpu().numpy()
    worst_q = worst_qd = worst_p = 0.0
    for k in range(0, n, 4):
        qo, qdo = dynamic_substeps(dyn, cfg, q0[k], qd0[k], act[k], env.r_lo, env.r_hi)
        worst_q = max(worst_q, np.abs(q1[k] - qo).max())
        worst_qd = max(worst_qd, np.abs(qd1[k] - qdo).max())
        worst_p = max(worst_p, np.abs(obs[k, 126:129].cpu().numpy() - fk_pointer(kin, qo)).max())
    assert worst_q <= 2e-5 and worst_qd <= 2e-4 and worst_p <= 5e-4, (worst_q, worst_qd, worst_p)
    # the observation carries q, qd and the applied action
    assert torch.equal(obs[:, 0:6], s["r"]) and torch.equal(obs[:, 90:96], s["v"])
    assert np.array_equal(obs[:, 108:114].cpu().numpy(), act)
    env.close()


def test_bounded_drift_over_1000_steps_under_pd_control():
    n = 64
    kw = dict(gravity=9.81, kp=2000.0, kd=500.0, torque_scale=1e5)
    env = make(n, seed=2, **kw)
    dyn, _ = chain_of(env)
    cfg = DynConfig(**kw)
    s = env.state()
    q, qd = s["r"].cpu().numpy().astype(np.float64), np.zeros((n, 6))
    rng = np.random.default_rng(1)
    worst = 0.0
    target = rng.uniform(env.r_lo * 0.8, env.r_hi * 0.8, size=(n, 6)).astype(np.float32)
    for t in range(1000):
        if t % 100 == 0:                                   # a new set point every 100 steps
            target = rng.uniform(env.r_lo * 0.8, env.r_hi * 0.8, size=(n, 6)).astype(np.float32)
        env.step_tensor(torch.as_tensor(target).cuda())
        for k in range(0, n, 16):                          # the float64 oracle free-runs beside 4 of the envs
            q[k], qd[k] = dynamic_substeps(dyn, cfg, q[k], qd[k], target[k], env.r_lo, env.r_hi)
        if t % 50 == 49 or t < 3:
            got = env.state()["r"].cpu().numpy()
            worst = max(worst, max(np.abs(got[k] - q[k]).max() for k in range(0, n, 16)))
    assert worst <= 2e-3, worst
    env.close()


def test_limits_reward_and_done_in_dynamic_mode():
    n = 256
    env = make(n, gravity=0.0, torque_scale=1e4, max_episode_steps=20, auto_reset=True, seed=8)
    push = torch.full((n, 6), 5e3, device="cuda")          # large torque into the upper limits
    r_hi = torch.as_tensor(env.r_hi).cuda()
    prev_pot = torch.zeros(n, device="cuda")
    for t in range(1, 41):
        obs, reward, flags = env.step_tensor(push)
        assert (obs[:, 0:6] <= r_hi).all()
        assert torch.allclose(reward, obs[:, 136] - prev_pot - 0.01, atol=1e-4)
        prev_pot = torch.where((flags & 1).bool(), torch.zeros_like(prev_pot), obs[:, 136])
        assert bool(((flags & 1) != 0).all()) == (t % 20 == 0)
    on = obs[:, 0:6] == r_hi
    assert on.any() and (obs[:, 90:96][on] == 0).all()     # stopped on the limit
    st = env.episode_stats()
    assert st["episodes"] == 2 * n and st["env_steps"] == 40 * n
    env.close()


def test_kinematic_mode_is_untouched_by_the_dynamic_fields():
    from pioneer_b200 import BatchConfig, BatchedPioneerEnv
    a = BatchedPioneerEnv(100, seed=1, batch_config=BatchConfig(kp=5.0, kd=1.0, torque_scale=3.0))
    b = BatchedPioneerEnv(100, seed=1)
    act = torch.rand((100, 6), device="cuda") * 50
    for _ in range(5):
        oa, ra, fa = a.step_tensor(act)
        ob, rb, fb = b.step_tensor(act)
        assert torch.equal(oa, ob) and torch.equal(ra, rb)
    a.close(); b.close()


def test_generic_chain_kernel_against_the_oracle(tmp_path):
    """A robot that is NOT the shipped axis pattern (tilted axis, rotated joint origin) takes the generic dynamics
    and kinematics code paths (runtime axis codes, Rodrigues rotation, origin rotation): same bars."""
    from pioneer_b200 import BatchConfig, BatchedPioneerEnv, SimulationConfig
    from pioneer_b200.urdf import DEFAULT_URDF
    text = open(DEFAULT_URDF).read()
    text = text.replace('<origin xyz="0 0 11"/><axis xyz="0 1 0"/>', '<origin xyz="0 0 11" rpy="0.3 -0.2 0.5"/><axis xyz="0 0.6 0.8"/>')
    text = text.replace('<origin xyz="11 0 0"/><axis xyz="0 1 0"/>', '<origin xyz="11 0 0"/><axis xyz="0 -1 0"/>')
    path = tmp_path / "tilted.urdf"
    path.write_text(text)
    n = 256
    kw = dict(gravity=9.81, kp=500.0, kd=100.0, torque_scale=1e4)
    env = BatchedPioneerEnv(n, urdf_path=str(path), seed=3, simulation_config=SimulationConfig(gravity=9.81),
                            batch_config=BatchConfig(mode="dynamic", kp=500.0, kd=100.0, torque_scale=1e4,
                                                     max_episode_steps=0, auto_reset=False))
    assert not np.allclose(env.chain.origin_rot[2], np.eye(3)) and np.allclose(env.chain.axis[2], (0, 0.6, 0.8))
    dyn, kin = chain_of(env)
    cfg = DynConfig(**kw)
    rng = np.random.default_rng(9)
    q0 = (rng.uniform(env.r_lo, env.r_hi, size=(n, 6)) * 0.7).astype(np.float32)
    qd0 = (rng.normal(size=(n, 6)) * 0.3).astype(np.float32)
    env.set_state(r=q0, v=qd0)
    act = rng.uniform(env.r_lo, env.r_hi, size=(n, 6)).astype(np.float32)
    obs, _, _ = env.step_tensor(torch.as_tensor(act).cuda())
    s = env.state()
    q1, qd1 = s["r"].cpu().numpy(), s["v"].cpu().numpy()
    for k in range(0, n, 8):
        qo, qdo = dynamic_substeps(dyn, cfg, q0[k], qd0[k], act[k], env.r_lo, env.r_hi)
        assert np.abs(q1[k] - qo).max() <= 2e-5 and np.abs(qd1[k] - qdo).max() <= 2e-4
        assert np.abs(obs[k, 126:129].cpu().numpy() - fk_pointer(kin, qo)).max() <= 5e-4
    env.close()
    # and the kinematic mode on the same robot: pointer position against the float64 FK
    kenv = BatchedPioneerEnv(n, urdf_path=str(path), seed=3, batch_config=BatchConfig(max_episode_steps=0, auto_reset=False))
    kenv.reset_world(q0, np.tile(np.array([[20, 0, 4]], np.float32), (n, 1)))
    o = kenv.step_tensor(torch.zeros((n, 6), device="cuda"))[0].cpu().numpy()
    for k in range(0, n, 8):
        assert np.abs(o[k, 126:129] - fk_pointer(kin, q0[k])).max() <= 2e-4
    kenv.close()


@pytest.mark.parametrize("chain", [0, 1])
def test_less_specialised_kernels_agree_with_the_shipped_one(tmp_path, chain):
    """The shipped URDF runs pnr_step_dynamic_kernel<..., PIONEER_ISO>; a modified copy of it selects a less specialised
    instantiation from the robot model alone.
    0, GENERIC (run-time axis codes): every joint limit widened to +-100 rad, beyond the +-64 rad of the PIONEER axis
    pattern, with the same physics.  From states and PD set points well inside the shipped limits no joint stop engages,
    so one env step from identical states lands within the float32-vs-float64 bar of the shipped kernel's.
    1, PIONEER (axis structure only): arm1's centre of mass moved off its frame origin, so the composite bodies are no
    longer isotropic.  The physics now differs from the shipped robot's: one env step is checked against the float64
    oracle with the bars of test_one_step_against_the_float64_oracle.
    (All three are checked against the oracle on the CPU in tests/test_dynamics_host.py.)"""
    import re
    from pioneer_b200.urdf import DEFAULT_URDF
    text = open(DEFAULT_URDF).read()
    if chain == 0:
        text, count = re.subn(r'lower="[^"]+" upper="[^"]+"', 'lower="-100" upper="100"', text)
    else:
        text, count = re.subn(r'(<link name="robot:arm1"><inertial>)', r'\1<origin xyz="0.5 0 4"/>', text)
    assert count == (6 if chain == 0 else 1)
    path = tmp_path / "less_specialised.urdf"
    path.write_text(text)
    n = 2048
    kw = dict(gravity=9.81, kp=800.0, kd=200.0, torque_scale=1e4)
    rng = np.random.default_rng(21)
    ref_env = make(n, seed=5, **kw)
    env = make(n, seed=5, urdf_path=str(path), **kw)
    q0 = rng.uniform(ref_env.r_lo * 0.5, ref_env.r_hi * 0.5, size=(n, 6)).astype(np.float32)
    qd0 = (rng.normal(size=(n, 6)) * 0.5).astype(np.float32)
    act = rng.uniform(ref_env.r_lo * 0.5, ref_env.r_hi * 0.5, size=(n, 6)).astype(np.float32)
    for e in (ref_env, env):
        e.set_state(r=q0, v=qd0)
        obs = e.step_tensor(torch.as_tensor(act).cuda())[0]
    ref, got = ref_env.state(), env.state()
    if chain == 0:
        assert (env.r_lo == -100).all() and (env.r_hi == 100).all()
        lo, hi = torch.as_tensor(ref_env.r_lo).cuda(), torch.as_tensor(ref_env.r_hi).cuda()
        assert ((ref["r"] > lo) & (ref["r"] < hi)).all()           # no joint stop engaged in either run
        assert (got["r"] - ref["r"]).abs().max().item() <= 2e-5
        assert (got["v"] - ref["v"]).abs().max().item() <= 2e-4
    else:
        assert np.abs(env.chain.body_com[1]).max() > 0
        dyn, kin = chain_of(env)
        cfg = DynConfig(**kw)
        q1, qd1 = got["r"].cpu().numpy(), got["v"].cpu().numpy()
        worst_q = worst_qd = worst_p = 0.0
        for k in range(0, n, 16):
            qo, qdo = dynamic_substeps(dyn, cfg, q0[k], qd0[k], act[k], env.r_lo, env.r_hi)
            worst_q = max(worst_q, np.abs(q1[k] - qo).max())
            worst_qd = max(worst_qd, np.abs(qd1[k] - qdo).max())
            worst_p = max(worst_p, np.abs(obs[k, 126:129].cpu().numpy() - fk_pointer(kin, qo)).max())
        assert worst_q <= 2e-5 and worst_qd <= 2e-4 and worst_p <= 5e-4, (worst_q, worst_qd, worst_p)
    ref_env.close(); env.close()
