"""Parity of the CUDA path (through the C-ABI, include/pioneer_b200.h) against
  * the golden vectors recorded from the unmodified reference source (tests/golden/make_golden.py), and
  * the CPU oracle (oracle/reach_oracle.py) on the same seeded inputs.

Bars (SURVEY.md 8(c)):
  * joint state r, v, a                : BIT-EXACT (explicitly rounded IEEE float32 arithmetic, no FMA)
  * done / truncated masks             : BIT-EXACT (the distance test is re-decided in float64 inside a band)
  * pointer xyz, distance              : |diff| <= 2e-4   (float32 FK at ~30-unit reach vs the reference's float64)
  * potential, reward                  : |diff| <= 1e-3   (d potential / d distance <= 9.5)
  * cos / sin observation columns      : |diff| <= 5e-7   (CUDA sincosf vs numpy float32 cos/sin, ~1 ulp each)
  * every other observation column     : BIT-EXACT
"""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle.reach_oracle import PNR_DONE, PNR_TRUNCATED
from tests._gpu import POS_COLS, POS_TOL, REW_TOL, TRIG_COLS, TRIG_TOL, VALUE_COLS, c_oracle_for, check_obs, kinematic_env
from tests._util import golden_case, load_golden

pytestmark = pytest.mark.gpu
G = load_golden()


def replay_golden(name, pioneer_config=None):
    """One env driven exactly like tests/golden/make_golden.py::rollout drove the reference."""
    case = golden_case(G, name)
    env = kinematic_env(1, max_episode_steps=500, auto_reset=False, **(pioneer_config or {}))
    ep = 0
    first = env.reset_world(case["q0"][ep][None], case["target"][ep][None], observe=True).cpu().numpy()[0]
    check_obs(first, case["reset_obs"][ep], f"{name} reset obs")
    obs_at = {int(t): k for k, t in enumerate(case["obs_idx"])}
    actions = torch.as_tensor(case["actions"]).cuda()
    for t in range(len(case["actions"])):
        obs, reward, flags = env.step_tensor(actions[t:t + 1])
        s = env.state()
        r, v, a = (s[k].cpu().numpy()[0] for k in ("r", "v", "a"))
        assert np.array_equal(r, case["r"][t]), (name, t, r, case["r"][t])
        assert np.array_equal(v, case["v"][t]), (name, t, v, case["v"][t])
        assert np.array_equal(a, case["a"][t]), (name, t)
        f = int(flags[0])
        assert bool(f & PNR_DONE) == bool(case["done"][t]), (name, t)
        assert bool(f & PNR_TRUNCATED) == bool(case["truncated"][t]), (name, t)
        o = obs.cpu().numpy()[0]
        np.testing.assert_allclose(o[126:136], case["tail"][t][:10], rtol=0, atol=POS_TOL, err_msg=f"{name} {t}")
        np.testing.assert_allclose(o[136], case["tail"][t][10], rtol=0, atol=REW_TOL)
        np.testing.assert_allclose(float(reward[0]), case["reward"][t], rtol=0, atol=REW_TOL, err_msg=f"{name} {t}")
        if t in obs_at:
            check_obs(o, case["obs"][obs_at[t]], f"{name} obs at {t}")
        if case["done"][t]:
            ep += 1
            first = env.reset_world(case["q0"][ep][None], case["target"][ep][None], observe=True).cpu().numpy()[0]
            check_obs(first, case["reset_obs"][ep], f"{name} reset obs {ep}")
    env.close()


@pytest.mark.parametrize("name", ["cfg1", "gentle", "bangbang", "wild", "zero", "reach", "approach"])
def test_golden_replay(name):
    replay_golden(name)


def test_golden_reward_knobs():
    replay_golden("knobs", dict(award_potential_slope=4.0, award_done=7.5, penalty_step=0.02))


def test_golden_multi_env_batch():
    """16 envs x 200 steps in ONE batch (a half-filled warp tile); env 0 is the cfg1 trajectory."""
    env = kinematic_env(16, max_episode_steps=500, auto_reset=False)
    env.reset_world(G["multi__q0"], G["multi__target"])
    actions = torch.as_tensor(G["multi__actions"]).cuda()
    for t in range(200):
        obs, reward, flags = env.step_tensor(actions[:, t].contiguous())
        s = env.state()
        assert np.array_equal(s["r"].cpu().numpy(), G["multi__r"][:, t]), t
        assert np.array_equal(s["v"].cpu().numpy(), G["multi__v"][:, t]), t
        np.testing.assert_allclose(reward.cpu().numpy(), G["multi__reward"][:, t], rtol=0, atol=REW_TOL)
        np.testing.assert_allclose(obs.cpu().numpy()[:, 126:136], G["multi__tail"][:, t, :10], rtol=0, atol=POS_TOL)
        assert np.array_equal((flags.cpu().numpy() & 1).astype(bool), G["multi__done"][:, t])
    env.close()


# ---------------------------------------------------------------------------------------------
# CUDA path vs CPU oracle on the same seeded inputs: Philox resets, auto-reset, both observation
# modes, both arithmetic modes, ragged batch sizes (not a multiple of the 32-env warp tile)
# ---------------------------------------------------------------------------------------------
def run_vs_oracle(n, steps, arith, obs_mode, max_episode_steps, seed, env_id_base=0, action_scale=1.0,
                  near_targets=False):
    env = kinematic_env(n, max_episode_steps=max_episode_steps, auto_reset=True, obs_mode=obs_mode, arith=arith,
                        seed=seed, env_id_base=env_id_base)
    ob = c_oracle_for(env, seed, compiled=False)
    # both sides were created reset with tick 0: same Philox draws
    s = env.state()
    os_ = ob.state()
    assert np.array_equal(s["r"].cpu().numpy(), os_["r"])
    assert np.array_equal(s["target"].cpu().numpy(), os_["target"].astype(np.float32))
    if near_targets:      # put every target within reach of the pointer so the distance-done path fires
        rng = np.random.default_rng(seed + 5)
        ptr = np.array([e.observe()[126:129] for e in ob.envs])
        tgt = (ptr + rng.normal(size=(n, 3)) * 0.08).astype(np.float32)
        q0 = os_["r"]
        ob.reset(q0=q0, target=tgt)
        env.reset_world(q0, tgt)
    check_obs(env.observe().cpu().numpy(), np.array([e.observe() for e in ob.envs]), "initial obs")
    rng = np.random.default_rng(seed + 1)
    a_max = env.a_max
    n_done = 0
    for t in range(steps):
        act = (rng.uniform(-1, 1, size=(n, 6)) * a_max * action_scale).astype(np.float32)
        obs, reward, flags = env.step_tensor(torch.as_tensor(act).cuda())
        o_obs, o_reward, o_flags = ob.step(act)
        assert np.array_equal(flags.cpu().numpy(), o_flags), f"done mask differs at step {t}"
        n_done += int((o_flags & 1).sum())
        s, os_ = env.state(), ob.state()
        for k in ("r", "v", "a"):
            assert np.array_equal(s[k].cpu().numpy(), os_[k]), f"{k} differs at step {t}"
        assert np.array_equal(s["t"].cpu().numpy(), os_["t"]), t
        assert np.array_equal(s["target"].cpu().numpy(), os_["target"].astype(np.float32)), t
        np.testing.assert_allclose(reward.cpu().numpy(), o_reward, rtol=0, atol=REW_TOL)
        np.testing.assert_allclose(s["ep_return"].cpu().numpy(), os_["ep_return"], rtol=0, atol=REW_TOL * (t + 2))
        check_obs(obs.cpu().numpy(), o_obs, f"step {t}")
    st = env.episode_stats()
    assert st["episodes"] == ob.stats[0] == n_done
    assert st["env_steps"] == ob.stats[6] == n * steps
    assert st["reached_target"] == ob.stats[7]
    if n_done:
        np.testing.assert_allclose(st["sum_return"], ob.stats[1], rtol=1e-5, atol=REW_TOL * steps)
        np.testing.assert_allclose(st["sum_length"], ob.stats[2])
        np.testing.assert_allclose([st["max_return"], st["min_return"]], ob.stats[4:6], atol=REW_TOL * steps)
    env.close()
    return n_done


@pytest.mark.parametrize("arith", ["f32", "legacy64"])
@pytest.mark.parametrize("obs_mode", ["terminal", "autoreset"])
def test_vs_oracle_random_rollout(arith, obs_mode):
    # TimeLimit 7 => every env auto-resets 3 times in 24 steps; 77 envs = 2 full warp tiles + a ragged one
    n_done = run_vs_oracle(77, 24, arith, obs_mode, max_episode_steps=7, seed=1234)
    assert n_done == 77 * 3


def test_vs_oracle_distance_done_and_autoreset():
    n_done = run_vs_oracle(40, 12, "f32", "terminal", max_episode_steps=500, seed=99, action_scale=0.002,
                           near_targets=True)
    assert n_done >= 10


def test_vs_oracle_sharded_ids():
    """env_id_base offsets the Philox counter: a shard starting at global id 1000 matches the oracle's."""
    run_vs_oracle(33, 10, "f32", "terminal", max_episode_steps=4, seed=7, env_id_base=1000)


def test_single_env_and_tiny_batches():
    for n in (1, 2, 31, 32, 33):
        run_vs_oracle(n, 3, "f32", "terminal", max_episode_steps=2, seed=n)


# ---------------------------------------------------------------------------------------------
# size-independent properties at BASELINE.json's full sizes (SURVEY.md 8(c) C6)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [4096, 65536])
def test_invariants_full_size(n):
    env = kinematic_env(n, max_episode_steps=500, auto_reset=True, seed=3)
    obs0 = env.reset()
    # (i) after reset: a = v = 0, potential = 0 -> obs[90:126] = {0,1,0,0,1,0} pattern, obs[136] = 0
    o = obs0.cpu().numpy()
    assert (o[:, 90:96] == 0).all() and (o[:, 96:102] == 1).all() and (o[:, 102:108] == 0).all()
    assert (o[:, 108:114] == 0).all() and (o[:, 114:120] == 1).all() and (o[:, 120:126] == 0).all()
    assert (o[:, 136] == 0).all()
    r_lo, r_hi, v_max = (torch.as_tensor(x).cuda() for x in (env.r_lo, env.r_hi, env.v_max))
    tlo, thi = (torch.tensor(x, dtype=torch.float32).cuda() for x in (env.config.target_lo, env.config.target_hi))
    assert ((obs0[:, 0:6] >= r_lo) & (obs0[:, 0:6] <= r_hi)).all()
    assert ((obs0[:, 129:132] >= tlo) & (obs0[:, 129:132] <= thi)).all()
    g = torch.Generator(device="cuda").manual_seed(0)
    a_max = torch.as_tensor(env.a_max).cuda()
    prev_pot = torch.zeros(n, device="cuda")
    prev_r = obs0[:, 0:6].clone()
    for t in range(1, 41):
        act = (torch.rand((n, 6), device="cuda", generator=g) * 2 - 1) * a_max
        if t == 1:
            act_first = act.clone()
        obs, reward, flags = env.step_tensor(act)
        r, v, a = obs[:, 0:6], obs[:, 90:96], obs[:, 108:114]
        # (iv) bounds; v == 0 exactly on a limit
        assert ((r >= r_lo) & (r <= r_hi)).all() and (v.abs() <= v_max).all()
        on_limit = (r == r_lo) | (r == r_hi)
        assert (v[on_limit] == 0).all()
        # (v) the action given at step t first moves the arm at step t+1
        if t == 1:
            assert torch.equal(r, prev_r)
        assert torch.equal(a, act)
        # (vi) obs[132:135] = target - pointer, obs[135] = norm
        diff = obs[:, 129:132] - obs[:, 126:129]
        assert torch.allclose(obs[:, 132:135], diff, atol=1e-5)
        assert torch.allclose(obs[:, 135], diff.double().norm(dim=1).float(), atol=1e-4)
        # (ii) reward = potential - old potential - 0.01 (+5): no env is done by distance here
        reached = (flags & PNR_DONE).bool() & ~(flags & PNR_TRUNCATED).bool()
        expect = obs[:, 136] - prev_pot - 0.01 + 5.0 * reached
        assert torch.allclose(reward, expect, atol=1e-4)
        pot = 95.0 / (obs[:, 135].double() / 10.0 + 1.0)
        assert torch.allclose(obs[:, 136].double(), pot, atol=1e-4)
        prev_pot = torch.where((flags & PNR_DONE).bool(), torch.zeros_like(prev_pot), obs[:, 136])
        # trig columns are the sin/cos of their value columns
        assert torch.allclose(obs[:, 6:12], torch.cos(r.double()).float(), atol=1e-6)
        assert torch.allclose(obs[:, 120:126], torch.sin(a.double()).float(), atol=1e-6)
    assert env.episode_stats()["env_steps"] == 40 * n
    env.close()


def test_time_limit_and_zero_action_properties():
    """(iii) a == 0 forever: r constant, reward == -0.01 from step 2 on; (vii) done at step 500 whatever the distance."""
    n = 4096
    env = kinematic_env(n, max_episode_steps=500, auto_reset=True, seed=11)
    obs0 = env.reset().clone()
    zero = torch.zeros((n, 6), device="cuda")
    for t in range(1, 501):
        obs, reward, flags = env.step_tensor(zero)
        if t == 2:
            assert torch.equal(obs[:, 0:6], obs0[:, 0:6])
            assert torch.allclose(reward, torch.full_like(reward, -0.01), atol=1e-6)
        if t < 500:
            assert int(flags.max()) == 0
    assert (flags == (PNR_DONE | PNR_TRUNCATED)).all()
    assert torch.equal(obs[:, 0:6], obs0[:, 0:6])            # terminal observation, not the reset one
    st = env.episode_stats()
    assert st["episodes"] == n and st["sum_length"] == 500 * n and st["reached_target"] == 0
    after = env.state()
    assert (after["t"] == 0).all() and not torch.equal(after["r"], obs0[:, 0:6])   # auto-reset drew new episodes
    env.close()


def test_sharding_is_invisible():
    """Two handles covering global ids [0, 3000) and [3000, 6000) reproduce one handle of 6000 envs bit for bit."""
    n = 6000
    whole = kinematic_env(n, max_episode_steps=5, seed=21)
    lo = kinematic_env(3000, max_episode_steps=5, seed=21, env_id_base=0)
    hi = kinematic_env(3000, max_episode_steps=5, seed=21, env_id_base=3000)
    g = torch.Generator(device="cuda").manual_seed(1)
    a_max = torch.as_tensor(whole.a_max).cuda()
    for t in range(12):
        act = (torch.rand((n, 6), device="cuda", generator=g) * 2 - 1) * a_max
        o, r, f = whole.step_tensor(act)
        o1, r1, f1 = lo.step_tensor(act[:3000].contiguous())
        o2, r2, f2 = hi.step_tensor(act[3000:].contiguous())
        assert torch.equal(o, torch.cat([o1, o2])) and torch.equal(r, torch.cat([r1, r2]))
        assert torch.equal(f, torch.cat([f1, f2]))
    a, b, c = whole.episode_stats(), lo.episode_stats(), hi.episode_stats()
    assert a["episodes"] == b["episodes"] + c["episodes"] == 2 * n
    for e in (whole, lo, hi):
        e.close()


def test_step_host_matches_step_tensor():
    n = 1000
    a_env = kinematic_env(n, max_episode_steps=6, seed=5)
    b_env = kinematic_env(n, max_episode_steps=6, seed=5)
    rng = np.random.default_rng(0)
    for t in range(8):
        act = (rng.uniform(-1, 1, size=(n, 6)) * a_env.a_max).astype(np.float32)
        o, r, f = a_env.step_tensor(torch.as_tensor(act).cuda())
        ho, hr, hf = b_env.step_host(act)
        assert np.array_equal(o.cpu().numpy(), ho) and np.array_equal(r.cpu().numpy(), hr)
        assert np.array_equal(f.cpu().numpy(), hf)
    a_env.close(); b_env.close()


def test_reset_subset_and_observe_indices():
    n = 100
    env = kinematic_env(n, max_episode_steps=0, auto_reset=False, seed=2)
    before = env.state()
    idx = [3, 50, 99]
    q0 = np.zeros((3, 6), np.float32)
    tg = np.array([[20, 0, 4]] * 3, np.float32)
    obs = env.reset_world(q0, tg, indices=idx, observe=True).cpu().numpy()
    np.testing.assert_allclose(obs[:, 126:129], [[14.6, 1.0, 15.9]] * 3, atol=1e-5)     # FK known answer, q = 0
    after = env.state()
    keep = np.setdiff1d(np.arange(n), idx)
    assert torch.equal(after["r"][keep], before["r"][keep])
    assert (after["r"][idx] == 0).all()
    assert np.array_equal(env.observe(indices=idx).cpu().numpy(), obs)
    env.close()


def test_fk_known_answers_on_device():
    """Hand-derived known answers, SURVEY.md section 8(c) C5, through pnr_reset + pnr_observe."""
    kat = {
        (0, 0, 0, 0, 0, 0): (14.6, 1.0, 15.9),
        (0.5, 0, 0, 0, 0, 0): (12.333279864995, 7.877195425512, 15.9),
        (0, 0.5, 0, 0, 0, 0): (18.997294851594, 1.0, 7.321202184764),
        (0, 0, 0.5, 0, 0, 0): (13.723613926947, 1.0, 8.667794003970),
        (0, 0, 0, 0.5, 0, 0): (14.6, 0.089091476652, 15.667406867592),
        (0, 0, 0, 0, 0.5, 0): (15.070205746153, 1.0, 13.941474928617),
        (0, 0, 0, 0, 0, 0.5): (14.6, 0.089091476652, 15.667406867592),
        (0.3, -0.4, 0.9, 1.1, -0.7, 2.0): (7.904033967723, 1.072102752440, 5.624962379045),
    }
    env = kinematic_env(len(kat), max_episode_steps=0, auto_reset=False)
    q = np.array(list(kat.keys()), np.float32)
    obs = env.reset_world(q, np.zeros((len(kat), 3), np.float32), observe=True).cpu().numpy()
    np.testing.assert_allclose(obs[:, 126:129], np.array(list(kat.values())), atol=2e-5)
    env.close()


def test_errors_are_loud():
    from pioneer_b200 import _cabi
    env = kinematic_env(8)
    with pytest.raises(_cabi.PioneerB200Error):
        _cabi.check(env._lib.pnr_step(env._h, None, None, None, None, None), "pnr_step")
    with pytest.raises(_cabi.PioneerB200Error):
        _cabi.check(env._lib.pnr_reset(env._h, None, 3, None, None, None, None), "pnr_reset")
    env.close()


# ---------------------------------------------------------------------------------------------
# BASELINE.json configs[1]: 4,096 envs on one B200, 1,000 steps, same seeds/actions as the CPU oracle (the C
# restatement, oracle/reach_oracle.c): per-step q / qdot / pointer diff, done/reset masks bit-exact.
# ---------------------------------------------------------------------------------------------
def test_cfg2_4096_envs_1000_steps_vs_c_oracle():
    n, steps, seed = 4096, 1000, 2026
    env = kinematic_env(n, max_episode_steps=500, auto_reset=True, obs_mode="terminal", seed=seed)
    cc = c_oracle_for(env, seed)
    rng = np.random.default_rng(7)
    worst = dict(pos=0.0, rew=0.0, trig=0.0)
    n_done = 0
    for t in range(steps):
        # mostly in-range random actions; every 50th step a burst far outside the action space (stored unclipped)
        scale = 40.0 if t % 50 == 49 else 1.0
        act = (rng.uniform(-1, 1, size=(n, 6)) * env.a_max * scale).astype(np.float32)
        obs, reward, flags = env.step_tensor(torch.as_tensor(act).cuda())
        o_obs, o_reward, o_flags = cc.step(act)
        assert np.array_equal(flags.cpu().numpy(), o_flags), f"done/reset mask differs at step {t}"
        n_done += int((o_flags & 1).sum())
        o = obs.cpu().numpy().astype(np.float64)
        assert np.array_equal(o[:, VALUE_COLS], o_obs[:, VALUE_COLS]), f"q / qdot / a / target differ at step {t}"
        worst["pos"] = max(worst["pos"], float(np.abs(o[:, POS_COLS] - o_obs[:, POS_COLS]).max()))
        worst["trig"] = max(worst["trig"], float(np.abs(o[:, TRIG_COLS] - o_obs[:, TRIG_COLS]).max()))
        worst["rew"] = max(worst["rew"], float(np.abs(reward.cpu().numpy() - o_reward).max()))
        if t % 100 == 99 or t == steps - 1:      # the internal state after auto-resets as well
            s, os_ = env.state(), cc.state()
            for k in ("r", "v", "a", "t"):
                assert np.array_equal(s[k].cpu().numpy(), os_[k]), (k, t)
    assert n_done == 2 * n                       # TimeLimit at steps 500 and 1000, Philox auto-resets in between
    assert worst["pos"] <= POS_TOL and worst["rew"] <= REW_TOL and worst["trig"] <= TRIG_TOL, worst
    st = env.episode_stats()
    assert st["episodes"] == cc.stats[0] and st["env_steps"] == n * steps
    np.testing.assert_allclose(st["sum_return"], cc.stats[1], rtol=1e-5)
    env.close()


@pytest.mark.parametrize("n", [262144 + 17, 1048576])
def test_deep_grid_stride_pipeline_vs_c_oracle(n):
    """Many tiles per CTA (the producer / consumer pipeline over two tile buffers runs 10-55 iterations deep):
    every row against the C oracle, plus run-to-run bit-identity of two handles (a barrier protocol error or a
    tile-buffer race would show up as a mismatch somewhere in 10^6 rows)."""
    seed, steps = 77, 3
    a = kinematic_env(n, max_episode_steps=2, auto_reset=True, obs_mode="terminal", seed=seed)
    b = kinematic_env(n, max_episode_steps=2, auto_reset=True, obs_mode="terminal", seed=seed)
    cc = c_oracle_for(a, seed)
    g = torch.Generator(device="cuda").manual_seed(5)
    a_max = torch.as_tensor(a.a_max).cuda()
    for t in range(steps):
        act = (torch.rand((n, 6), device="cuda", generator=g) * 2 - 1) * a_max
        oa, ra, fa = a.step_tensor(act)
        ob, rb, fb = b.step_tensor(act)
        assert torch.equal(oa, ob) and torch.equal(ra, rb) and torch.equal(fa, fb), t
        o_obs, o_rew, o_flags = cc.step(act.cpu().numpy())
        assert np.array_equal(fa.cpu().numpy(), o_flags), t
        o = oa.cpu().numpy().astype(np.float64)
        assert np.array_equal(o[:, VALUE_COLS], o_obs[:, VALUE_COLS]), t
        assert np.abs(o[:, POS_COLS] - o_obs[:, POS_COLS]).max() <= POS_TOL
        assert np.abs(o[:, TRIG_COLS] - o_obs[:, TRIG_COLS]).max() <= TRIG_TOL
        assert np.abs(ra.cpu().numpy() - o_rew).max() <= REW_TOL
    sa, sc = a.state(), cc.state()
    for k in ("r", "v", "a", "t"):
        assert np.array_equal(sa[k].cpu().numpy(), sc[k]), k
    a.close(); b.close()


def test_non_finite_and_degenerate_actions_follow_the_reference_arithmetic():
    """The reference stores the action unclipped (pioneer_knm_env.py:144) and feeds it to the next step's integrator:
    NaN propagates through every comparison, +-inf saturates the velocity with a zero first phase, a = -eps makes the
    divisor of the saturation time exactly zero.  Same bits as the oracle, NaN for NaN."""
    n = 64
    env = kinematic_env(n, max_episode_steps=0, auto_reset=False, seed=8)
    ob = c_oracle_for(env, 8, compiled=False)
    rng = np.random.default_rng(0)
    eps32 = np.float32(1e-5)
    specials = np.array([np.nan, np.inf, -np.inf, 3e38, -3e38, -eps32, 0.0, -0.0, 1e-40, 1.2e5, -1.2e5], np.float32)
    for t in range(8):
        act = (rng.uniform(-1, 1, size=(n, 6)) * env.a_max).astype(np.float32)
        if t in (1, 4):                                       # sprinkle the special values over the batch
            pick = rng.integers(0, len(specials), size=(n, 6))
            mask = rng.random((n, 6)) < 0.5
            act = np.where(mask, specials[pick], act).astype(np.float32)
        with np.errstate(all="ignore"):
            o_obs, o_rew, o_flags = ob.step(act)
        obs, rew, flags = env.step_tensor(torch.as_tensor(act).cuda())
        s, os_ = env.state(), ob.state()
        for k in ("r", "v", "a"):
            got, want = s[k].cpu().numpy(), os_[k]
            assert np.array_equal(got, want, equal_nan=True), (k, t)
            assert np.array_equal(np.signbit(got[want == 0]), np.signbit(want[want == 0])), (k, t)   # signed zeros too
        assert np.array_equal(flags.cpu().numpy(), o_flags), t
        o = obs.cpu().numpy().astype(np.float64)
        # NaN exactly where the reference has it -- except that the oracle's Rodrigues FK turns the WHOLE pointer into
        # NaN when one joint angle is NaN, while the kernel's axis-aligned rotations leave the coordinate along that
        # axis finite (distance, potential and reward are NaN on both sides)
        strict = np.r_[0:126, 129:132, 135:137]
        assert np.array_equal(np.isnan(o[:, strict]), np.isnan(o_obs[:, strict])), t
        loose = np.r_[126:129, 132:135]
        assert not (np.isnan(o[:, loose]) & ~np.isnan(o_obs[:, loose])).any(), t
        o_obs = np.where(np.isnan(o), np.nan, o_obs)
        o = np.where(np.isnan(o_obs), np.nan, o)
        inf = np.isinf(o_obs)
        assert np.array_equal(o[inf], o_obs[inf]), t                                 # +-inf where the reference has it
        fin = np.isfinite(o_obs)
        tol = 1e-3 + 1e-6 * np.abs(o_obs[fin])                                      # stored actions reach 3e38
        assert (np.abs(o[fin] - o_obs[fin]) <= tol).all(), t
        assert np.array_equal(np.isnan(rew.cpu().numpy()), np.isnan(o_rew))
    assert np.isnan(env.state()["r"].cpu().numpy()).any() and np.isfinite(env.state()["r"].cpu().numpy()).any()
    env.close()


@pytest.mark.parametrize("case", range(4))
def test_randomised_configs_vs_c_oracle(case):
    """Every knob of PioneerKinematicConfig / SimulationConfig / TimeLimit travels through pnr_config into the kernel:
    randomised settings (limits ratios, done distance, reward shaping, target box, timestep, frame_skip) against the C
    oracle on the same seeds and actions."""
    from pioneer_b200 import BatchConfig, BatchedPioneerEnv, PioneerKinematicConfig, SimulationConfig
    rng = np.random.default_rng(1000 + case)
    lo = rng.uniform([-5, -12, 0], [10, -2, 3])
    hi = lo + rng.uniform(1, 12, size=3)
    kw = dict(max_v_to_r=float(rng.uniform(0.5, 4)), max_a_to_v=float(rng.uniform(2, 20)),
              done_distance=float(rng.uniform(0.05, 6.0)), award_max=float(rng.uniform(50, 200)),
              award_done=float(rng.uniform(0, 20)), award_potential_slope=float(rng.uniform(2, 30)),
              penalty_step=float(rng.uniform(0, 0.1)), target_lo=tuple(lo), target_hi=tuple(hi))
    timestep, frame_skip, limit = float(rng.uniform(1 / 480, 1 / 60)), int(rng.integers(1, 20)), int(rng.integers(3, 12))
    n, seed = 2048 + case, 40 + case
    env = BatchedPioneerEnv(n, seed=seed, env_id_base=5 * case, pioneer_config=PioneerKinematicConfig(**kw),
                            simulation_config=SimulationConfig(timestep=timestep, frame_skip=frame_skip),
                            batch_config=BatchConfig(max_episode_steps=limit))
    cc = c_oracle_for(env, seed)
    assert np.array_equal(env.a_max, cc.a_max) and np.array_equal(env.v_max, cc.v_max)
    reached = 0
    for t in range(30):
        act = (rng.uniform(-1, 1, size=(n, 6)) * env.a_max).astype(np.float32)
        obs, rew, flags = env.step_tensor(torch.as_tensor(act).cuda())
        o_obs, o_rew, o_flags = cc.step(act)
        assert np.array_equal(flags.cpu().numpy(), o_flags), (case, t)
        reached += int(((o_flags & 1) != 0).sum() - ((o_flags & 2) != 0).sum())
        o = obs.cpu().numpy().astype(np.float64)
        assert np.array_equal(o[:, VALUE_COLS], o_obs[:, VALUE_COLS]), (case, t)
        assert np.abs(o[:, POS_COLS] - o_obs[:, POS_COLS]).max() <= POS_TOL
        assert np.abs(rew.cpu().numpy() - o_rew).max() <= REW_TOL * max(1.0, kw["award_max"] / 100)
    st = env.episode_stats()
    assert st["episodes"] == cc.stats[0] and st["reached_target"] == cc.stats[7]
    env.close()
