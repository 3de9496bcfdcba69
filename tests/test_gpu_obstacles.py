"""Reach-with-obstacles variant (BASELINE.json configs[3]): link capsules against the ground plane, the reference
demo's box (half extents (0.5, 0.5, 5) at (10, 5, 0), pioneer_knm_env.py:249-255) and a sphere.  The reference
robot has no collision geometry (0 <collision> elements) and no contact term in its reward: this variant is the
repo's extension, PARITY UNPINNED; the CUDA path is checked against oracle/reach_oracle.py::contact_depth."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle.reach_oracle import OracleChain, OracleConfig, OracleEnv, contact_depth
from pioneer_b200 import demo_obstacles
from tests._gpu import PENALTY, c_oracle_for, host_boxes, kinematic_env

pytestmark = pytest.mark.gpu


def make(n, obstacles, penalty=PENALTY, mode="kinematic", **kw):
    from pioneer_b200 import BatchConfig, BatchedPioneerEnv
    bc = BatchConfig(obstacles=obstacles, contact_penalty=penalty, mode=mode, max_episode_steps=kw.pop("max_episode_steps", 0),
                     auto_reset=kw.pop("auto_reset", False), torque_scale=kw.pop("torque_scale", 1.0))
    return BatchedPioneerEnv(n, batch_config=bc, **kw)


def oracle_obstacles(obs_list):
    return tuple((o.kind, o.position, o.extent) for o in obs_list)


def test_capsules_come_from_the_asset():
    from pioneer_b200.urdf import flatten_urdf
    m = flatten_urdf()
    assert len(m.capsules) == 5 and [c[0] for c in m.capsules] == [1, 2, 3, 4, 5]
    # arm1: 11 long along z of frame 1; effector capsule ends on the pointer
    assert np.allclose(m.capsules[0][2], (0, 0, 0)) and np.allclose(m.capsules[0][3], (0, 0, 11))
    assert np.allclose(m.capsules[4][3], m.tip_xyz)


@pytest.mark.parametrize("mode", ["kinematic", "dynamic"])
def test_contact_penalty_matches_the_oracle(mode):
    n = 96
    obstacles = demo_obstacles()
    plain = make(n, [], penalty=0.0, mode=mode, seed=5, torque_scale=50.0)
    env = make(n, obstacles, mode=mode, seed=5, torque_scale=50.0)
    chain = OracleChain.from_model(env.chain)
    rng = np.random.default_rng(0)
    hits = 0
    for t in range(12):
        act = (rng.uniform(-1, 1, size=(n, 6)) * env.a_max * (1.0 if mode == "kinematic" else 0.2)).astype(np.float32)
        a = torch.as_tensor(act).cuda()
        o1, r1, f1 = plain.step_tensor(a)
        o2, r2, f2 = env.step_tensor(a)
        assert torch.equal(o1, o2) and torch.equal(f1, f2)            # the obstacles only touch the reward
        q = o2[:, 0:6].cpu().numpy()
        depth = np.array([contact_depth(chain, q[k], oracle_obstacles(obstacles)) for k in range(n)])
        hits += int((depth > 0).sum())
        np.testing.assert_allclose((r1 - r2).cpu().numpy(), PENALTY * depth, rtol=0, atol=2e-3)
    assert hits > n                                                   # the arm really is in contact often
    plain.close(); env.close()


def test_each_obstacle_kind_known_answers():
    """q = 0: arm1 stands on z in [3, 14] at x = y = 0; arm2 runs along x at z = 14, y = 1."""
    from pioneer_b200 import Obstacle
    cases = [
        # plane z = 5 (normal +z): arm1's lower end (z = 3, radius 0.9) is 2 below it -> depth 2.9
        ([Obstacle("plane", (0, 0, 5), (0, 0, 1))], None),
        # sphere radius 1 centred 1.5 beside arm1's axis: depth 0.9 + 1 - 1.5 = 0.4 on arm1 only
        ([Obstacle("sphere", (1.5, 0, 8), (1.0, 0, 0))], 0.4),
        # box whose face is 0.5 from arm1's axis: depth 0.9 - 0.5 = 0.4
        ([Obstacle("box", (2.5, 0, 8), (2.0, 5.0, 1.0))], None),
        # far away: nothing
        ([Obstacle("sphere", (100, 100, 100), (1.0, 0, 0)), Obstacle("plane", (0, 0, -50), (0, 0, 1))], 0.0),
        # a THIN box (1 wide, the demo box's footprint) crossed by arm2 (x from 0 to 9 at y = 1, z = 14, radius 0.9) between
        # two of the former 8 sample points (x = 3.86 and 5.14): the axis passes through the box centre line, 0.5 deep,
        # so the exact depth is 0.9 + 0.5 = 1.4 (the 8-sample rule saw 0.9 - 0.14 = 0.76)
        ([Obstacle("box", (4.5, 1.0, 14.0), (0.5, 0.5, 5.0))], 1.4),
    ]
    for obstacles, expect in cases:
        env = make(4, obstacles, penalty=1.0)
        plain = make(4, [], penalty=0.0)
        q0 = np.zeros((4, 6), np.float32)
        tg = np.tile(np.array([[20, 0, 4]], np.float32), (4, 1))
        env.reset_world(q0, tg); plain.reset_world(q0, tg)
        zero = torch.zeros((4, 6), device="cuda")
        _, r2, _ = env.step_tensor(zero)
        _, r1, _ = plain.step_tensor(zero)
        depth = float((r1 - r2)[0])
        want = contact_depth(OracleChain.from_model(env.chain), q0[0], oracle_obstacles(obstacles))
        assert abs(depth - want) < 1e-4, (obstacles, depth, want)
        if expect is not None:
            assert abs(want - expect) < 1e-6, (obstacles, want, expect)
        env.close(); plain.close()


def test_box_distance_is_exact_between_the_former_sample_points():
    """arm2 straddling the thin box above: the exact rule sees the full penetration, and sliding the box along the link
    changes nothing (an 8-sample rule would oscillate with the box position)."""
    from pioneer_b200 import Obstacle
    depths = []
    for x in np.linspace(3.0, 7.5, 10):
        obstacles = [Obstacle("box", (float(x), 1.0, 14.0), (0.5, 0.5, 5.0))]
        env, plain = make(2, obstacles, penalty=1.0), make(2, [], penalty=0.0)
        q0, tg = np.zeros((2, 6), np.float32), np.tile(np.array([[20, 0, 4]], np.float32), (2, 1))
        env.reset_world(q0, tg); plain.reset_world(q0, tg)
        zero = torch.zeros((2, 6), device="cuda")
        depths.append(float((plain.step_tensor(zero)[1] - env.step_tensor(zero)[1])[0]))
        want = contact_depth(OracleChain.from_model(env.chain), q0[0], oracle_obstacles(obstacles))
        assert abs(depths[-1] - want) < 1e-4
        env.close(); plain.close()
    assert max(depths) - min(depths) < 1e-4 and abs(depths[0] - 1.4) < 1e-4, depths


@pytest.mark.parametrize("random_box", [False, True])
def test_config4_16384_envs_against_the_compiled_oracle(random_box):
    """BASELINE.json configs[3] in the kinematic mode: 16,384 envs x 60 steps with TimeLimit 25 (two auto-resets, which
    redraw the per-env box when random_box is on) against oracle/reach_oracle.c: joint state and flags bit-exact, reward
    (which carries the contact penalty) within 2e-3."""
    n = 16384
    env = kinematic_env(n, obstacles=True, random_box=random_box, max_episode_steps=25, auto_reset=True, seed=77)
    orc = c_oracle_for(env, 77)
    if random_box:
        assert np.array_equal(host_boxes(env), orc.boxes())
    rng = np.random.default_rng(3)
    worst = 0.0
    for t in range(60):
        act = (rng.uniform(-1, 1, size=(n, 6)) * env.a_max).astype(np.float32)
        obs, reward, flags = env.step_tensor(torch.as_tensor(act).cuda())
        _, o_reward, o_flags = orc.step(act, want_obs=False)
        assert np.array_equal(flags.cpu().numpy(), o_flags)
        worst = max(worst, float(np.abs(reward.cpu().numpy() - o_reward).max()))
    s, o = env.state(), orc.state()
    assert np.array_equal(s["r"].cpu().numpy(), o["r"]) and np.array_equal(s["v"].cpu().numpy(), o["v"])
    assert worst <= 2e-3, worst
    if random_box:
        assert np.array_equal(host_boxes(env), orc.boxes())
    st = env.episode_stats()
    assert st["episodes"] == orc.stats[0] == 2 * n
    env.close()


def test_oracle_env_applies_the_penalty():
    """The CPU oracle on its own, so both of its configurations are written by hand."""
    from pioneer_b200.urdf import flatten_urdf
    chain = OracleChain.from_model(flatten_urdf())
    obstacles = oracle_obstacles(demo_obstacles())
    a = OracleEnv(chain, OracleConfig())
    b = OracleEnv(chain, OracleConfig(obstacles=obstacles, contact_penalty=2.0))
    rng = np.random.default_rng(0)
    q0 = next(q for q in (rng.uniform(chain.lower, chain.upper).astype(np.float32) for _ in range(1000))
              if contact_depth(chain, q, obstacles) > 0.1)
    tg = (20.0, 0.0, 4.0)
    a.reset_world(q0, tg); b.reset_world(q0, tg)
    ra, _ = a.act(np.zeros(6, np.float32))
    rb, _ = b.act(np.zeros(6, np.float32))
    assert abs((ra - rb) - 2.0 * contact_depth(chain, q0, obstacles)) < 1e-12 and ra > rb


def test_config4_16384_envs_invariants():
    """BASELINE.json configs[3]: 16,384 envs with ground / box / sphere; penalty >= 0, zero weight == no obstacles."""
    n = 16384
    obstacles = demo_obstacles()
    env = make(n, obstacles, seed=1, max_episode_steps=500, auto_reset=True)
    off = make(n, obstacles, penalty=0.0, seed=1, max_episode_steps=500, auto_reset=True)
    plain = make(n, [], penalty=0.0, seed=1, max_episode_steps=500, auto_reset=True)
    g = torch.Generator(device="cuda").manual_seed(0)
    a_max = torch.as_tensor(env.a_max).cuda()
    total = 0.0
    for t in range(30):
        act = (torch.rand((n, 6), device="cuda", generator=g) * 2 - 1) * a_max
        o1, r1, f1 = plain.step_tensor(act)
        o2, r2, f2 = off.step_tensor(act)
        o3, r3, f3 = env.step_tensor(act)
        assert torch.equal(r1, r2) and torch.equal(o1, o2) and torch.equal(o1, o3)
        pen = r1 - r3
        assert (pen >= -1e-4).all()
        total += float(pen.sum())
    assert total > 0
    for e in (env, off, plain):
        e.close()
