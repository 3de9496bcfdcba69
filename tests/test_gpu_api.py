"""The reference-facing Python surface on the GPU: the single-env facade with the reference's constructor and
gym.Env contract (pioneer/envs/pioneer/pioneer_knm_env.py:38-242), the launcher's env factories
(pioneer/launch/pioneer_knm_train.py:20-29), the RLlib-style VectorEnv adapter and the CUDA-graph rollout."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from tests._gpu import dynamic_env, fragments_equal_single_steps, kinematic_env, uniform_actions
from tests._util import golden_case, load_golden

pytestmark = pytest.mark.gpu
G = load_golden()


def test_facade_has_the_reference_surface():
    from pioneer_b200.envs.pioneer import PioneerKinematicConfig, PioneerKinematicEnv
    env = PioneerKinematicEnv(headless=True, pioneer_config=PioneerKinematicConfig(), simulation_config=None,
                              render_config=None)
    assert env.dof == 6 and env.metadata["video.frames_per_second"] == 24
    assert np.array_equal(env.r_lo, G["const_r_lo"]) and np.array_equal(env.r_hi, G["const_r_hi"])
    assert np.array_equal(env.v_max, G["const_v_max"]) and np.array_equal(env.a_max, G["const_a_max"])
    assert env.dt == G["const_dt_eps"][0] and env.eps == G["const_dt_eps"][1]
    assert np.array_equal(env.action_space.low, G["const_action_low"])
    assert np.array_equal(env.action_space.high, G["const_action_high"])
    assert env.observation_space.shape == (137,) and str(env.observation_space.dtype) == "float64"
    assert [j.name for j in env.scene.joints] == list(G["const_joint_names"])
    assert set(G["const_item_names"]) <= set(env.scene.items_by_name)
    lo, hi = env.joint_limits()
    assert lo.dtype == np.float32 and np.array_equal(lo, G["const_r_lo"]) and np.array_equal(hi, G["const_r_hi"])
    np.testing.assert_allclose([env.compute_potential(d) for d in (0.0, 0.1, 5.0, 20.0)], G["const_potential_kat"])
    obs = env.reset()
    assert obs.shape == (137,) and obs.dtype == np.float64
    assert env.potential == 0 and (env.a == 0).all() and (env.v == 0).all()
    obs2, reward, done, info = env.step(env.action_space.sample())
    assert obs2.shape == (137,) and isinstance(reward, float) and isinstance(done, bool)
    assert set(info) == {"r_pot", "r_step", "r_done", "rw", "dist", "pot", "a", "v", "r"}      # pioneer_knm_env.py:167-179
    assert all(isinstance(v, str) for v in info.values())
    with pytest.raises(NotImplementedError):
        env.render()
    env.close()


def test_facade_under_timelimit_replays_the_reference_trajectory():
    """TimeLimit(PioneerKinematicEnv(cfg), 500) exactly as the reference launcher builds it, driven with the cfg1
    actions: joint state bit-exact, rewards/pointer within float32 tolerance, truncation at step 500."""
    from pioneer_b200.launch import prepare_env
    case = golden_case(G, "cfg1")
    tl = prepare_env({"award_potential_slope": 10.0, "award_done": 5.0, "penalty_step": 1 / 100})
    assert tl._max_episode_steps == 500
    env = tl.env
    tl.reset()
    env.reset_world(joint_positions=case["q0"][0], target_position=tuple(case["target"][0]))
    for t in range(510):
        obs, reward, done, info = tl.step(case["actions"][t])
        assert np.array_equal(env.r, case["r"][t]) and np.array_equal(env.v, case["v"][t]), t
        np.testing.assert_allclose(reward, case["reward"][t], atol=1e-3)
        np.testing.assert_allclose(obs[126:136], case["tail"][t][:10], atol=2e-4)
        assert done == bool(case["done"][t])
        assert bool(info.get("TimeLimit.truncated", False)) == bool(case["truncated"][t])
        if done:
            tl.reset()
            env.reset_world(joint_positions=case["q0"][1], target_position=tuple(case["target"][1]))
    tl.close()


def test_facade_seed_reproduces_the_reference_draw_order():
    """reset_world() draws 6 joint angles then 3 target coordinates from the env's RandomState (pioneer_knm_env.py:80-90)."""
    from pioneer_b200.envs.pioneer import PioneerKinematicEnv
    env = PioneerKinematicEnv()
    env.seed(123)
    obs = env.reset()
    rs = np.random.RandomState(123)
    q = rs.uniform(env.r_lo, env.r_hi)
    tgt = rs.uniform(np.array(env.config.target_lo), np.array(env.config.target_hi))
    assert np.array_equal(obs[0:6], q.astype(np.float32).astype(np.float64))
    assert np.array_equal(obs[129:132], tgt.astype(np.float32).astype(np.float64))
    env.close()


def test_facade_after_a_seeded_reset_replays_the_reference_bit_for_bit():
    """Golden case 'sampled': env.seed(123); env.reset() run by the unmodified reference (float64 start angles), 90 steps,
    a second seeded reset at step 40.  The facade draws with the same generator, hands the device float32(start), and the
    joint state is bit-equal from the first step on (see test_sampled_reset_keeps_float64... for why nothing is lost)."""
    from pioneer_b200.launch import prepare_env
    case = golden_case(G, "sampled")
    tl = prepare_env({"award_potential_slope": 10.0, "award_done": 5.0, "penalty_step": 1 / 100})
    env = tl.env
    env.seed(int(case["seed"]))
    ep = 0
    for t, action in enumerate(case["actions"]):
        if t in case["reset_at"]:
            obs0 = tl.reset()
            np.testing.assert_allclose(obs0[:126], case["reset_obs"][ep][:126], rtol=0, atol=6e-7)
            np.testing.assert_allclose(obs0[126:136], case["reset_obs"][ep][126:136], rtol=0, atol=2e-4)
            ep += 1
        obs, reward, done, info = tl.step(action)
        assert np.array_equal(env.r, case["r"][t]) and np.array_equal(env.v, case["v"][t]), t
        np.testing.assert_allclose(reward, case["reward"][t], atol=1e-3)
        np.testing.assert_allclose(obs[126:136], case["tail"][t][:10], atol=2e-4)
    tl.close()


def test_vector_env_rllib_contract():
    from pioneer_b200 import PioneerVectorEnv
    n = 48
    venv = PioneerVectorEnv(n, max_episode_steps=3, seed=9)
    obs = venv.vector_reset()
    assert isinstance(obs, list) and len(obs) == n and obs[0].shape == (137,)
    assert len(venv.get_unwrapped()) == n
    rng = np.random.default_rng(0)
    for t in range(1, 8):
        actions = [(rng.uniform(-1, 1, size=6) * venv.batch.a_max).astype(np.float32) for _ in range(n)]
        obs, rewards, dones, infos = venv.vector_step(actions)
        assert len(obs) == len(rewards) == len(dones) == len(infos) == n
        assert isinstance(rewards[0], float) and isinstance(dones[0], bool)
        if t % 3 == 0:
            assert all(dones) and all(i["TimeLimit.truncated"] for i in infos)
            terminal_r = np.array([o[0:6] for o in obs])
            # RLlib now calls reset_at(i): the kernel already started the next episode, its first observation comes back
            fresh = np.array([venv.reset_at(i) for i in range(n)])
            assert (fresh[:, 136] == 0).all() and (fresh[:, 90:96] == 0).all()
            assert not np.array_equal(fresh[:, 0:6], terminal_r)
            state_r = venv.batch.state()["r"].cpu().numpy()
            assert np.array_equal(fresh[:, 0:6], state_r)
        else:
            assert not any(dones) and all(i == {} for i in infos)
    # an explicit reset_at of an env that is NOT done starts a new episode for that env only
    before = venv.batch.state()["t"].cpu().numpy().copy()
    first = venv.reset_at(5)
    after = venv.batch.state()["t"].cpu().numpy()
    assert after[5] == 0 and first[136] == 0 and np.array_equal(np.delete(after, 5), np.delete(before, 5))
    venv.close()


def test_prepare_vector_env_factory():
    from pioneer_b200.launch import prepare_vector_env
    venv = prepare_vector_env({"award_potential_slope": 4.0, "award_done": 7.5, "penalty_step": 0.02, "num_envs": 64,
                               "seed": 1, "worker_index": 2})
    assert venv.num_envs == 64 and venv.batch.env_id_base == 128
    assert venv.batch.config.award_done == 7.5 and venv.batch.batch_config.max_episode_steps == 500
    venv.close()


def test_cuda_graph_rollout_equals_stepping():
    from pioneer_b200 import BatchConfig, BatchedPioneerEnv
    n, T, limit = 3000, 6, 4
    a = BatchedPioneerEnv(n, seed=4, batch_config=BatchConfig(max_episode_steps=limit))
    b = BatchedPioneerEnv(n, seed=4, batch_config=BatchConfig(max_episode_steps=limit))
    g = torch.Generator(device="cuda").manual_seed(0)
    actions = (torch.rand((T, n, 6), device="cuda", generator=g) * 2 - 1) * torch.as_tensor(a.a_max).cuda()
    obs = torch.zeros((T, n, 137), device="cuda")
    rew = torch.zeros((T, n), device="cuda")
    flg = torch.zeros((T, n), dtype=torch.uint8, device="cuda")
    # capture_rollout runs one eager step first (kernel attribute set-up); mirror it on the twin
    graph = a.capture_rollout(actions, obs, rew, flg)
    b.step_tensor(actions[0])
    graph.replay()
    torch.cuda.synchronize()
    for t in range(T):
        o, r, f = b.step_tensor(actions[t])
        assert torch.equal(f, flg[t]), t                                # TimeLimit flags never depend on the reset draws
        if t < limit - 1:                                                # the eager step + these: nobody has restarted yet
            assert torch.equal(r, rew[t]) and torch.equal(o, obs[t]), t
    # envs that restarted INSIDE the graph drew from the graph's own reset-key domain: valid states, different from the
    # eager twin's draws (eager steps and graph replays can be interleaved without ever reusing a reset key)
    sa, sb = a.state(), b.state()
    lo, hi = torch.as_tensor(a.r_lo).cuda(), torch.as_tensor(a.r_hi).cuda()
    assert (sa["r"] >= lo).all() and (sa["r"] <= hi).all() and torch.equal(sa["t"], sb["t"])
    assert (sa["target"] != sb["target"]).any(dim=1).float().mean() > 0.99
    a.close(); b.close()


def test_eager_steps_and_graph_replays_never_reuse_a_reset_key():
    """ADVICE r1: with the host counter frozen into the graph, an eager step after replay 1 and the first captured step of
    replay 2 used to draw the same (q, target).  Every step ends an episode here, so every step exposes its reset draw."""
    from pioneer_b200 import BatchConfig, BatchedPioneerEnv
    n, T = 256, 2
    env = BatchedPioneerEnv(n, seed=8, batch_config=BatchConfig(max_episode_steps=1))
    actions = torch.zeros((T, n, 6), device="cuda")
    obs = torch.zeros((T, n, 137), device="cuda")
    rew = torch.zeros((T, n), device="cuda")
    flg = torch.zeros((T, n), dtype=torch.uint8, device="cuda")
    graph = env.capture_rollout(actions, obs, rew, flg)
    seen = []

    def snap():
        torch.cuda.synchronize()
        seen.append(env.state()["target"].clone())

    for k in range(3):                      # replay, two eager steps, replay, ...
        graph.replay(); snap()
        env.step_tensor(actions[0]); snap()
        env.step_tensor(actions[0]); snap()
    # a second graph on the same handle gets its own domain
    graph2 = env.capture_rollout(actions, obs, rew, flg); snap()
    graph2.replay(); snap()
    graph.replay(); snap()
    for i in range(len(seen)):
        for j in range(i + 1, len(seen)):
            assert (seen[i] != seen[j]).any(dim=1).float().mean() > 0.99, (i, j)
    env.close()


def test_seed_reaches_steps_already_captured_in_a_graph():
    from pioneer_b200 import BatchConfig, BatchedPioneerEnv
    n, T = 256, 1
    env = BatchedPioneerEnv(n, seed=8, batch_config=BatchConfig(max_episode_steps=1))
    twin = BatchedPioneerEnv(n, seed=8, batch_config=BatchConfig(max_episode_steps=1))
    bufs = lambda: (torch.zeros((T, n, 6), device="cuda"), torch.zeros((T, n, 137), device="cuda"),
                    torch.zeros((T, n), device="cuda"), torch.zeros((T, n), dtype=torch.uint8, device="cuda"))
    g1, g2 = env.capture_rollout(*bufs()), twin.capture_rollout(*bufs())
    twin.seed(99)                           # after capture
    g1.replay(); g2.replay(); torch.cuda.synchronize()
    assert (env.state()["target"] != twin.state()["target"]).any(dim=1).float().mean() > 0.99
    assert twin.state_dict()["seed"] == 99
    env.close(); twin.close()


@pytest.mark.parametrize("mode,n", [("kinematic", 5000), ("kinematic", 37), ("kinematic", 4097), ("kinematic", 70001),
                                    ("kinematic", 300000), ("dynamic", 70001), ("dynamic", 2048), ("dynamic", 131072)])
def test_step_many_equals_stepping(mode, n):
    """pnr_step_many gives bit for bit what T separate pnr_step calls give, call after call.  The fragment is ONE launch:
    every CTA (kinematic mode; a CTA barrier between the steps) or warp (dynamic mode; env state in registers) runs the T
    steps on its own tiles -- incl. ragged last tiles, several tiles per CTA / warp, auto-resets between the steps."""
    from pioneer_b200 import _cabi
    make = kinematic_env if mode == "kinematic" else dynamic_env
    a, b = make(n, max_episode_steps=5, seed=4), make(n, max_episode_steps=5, seed=4)
    g = torch.Generator(device="cuda").manual_seed(0)
    fragments_equal_single_steps(a, b, T=7 if n < 200000 else 3, fragments=4 if n < 200000 else 2, generator=g,
                                 return_rtol=0)
    # T = 0 launches nothing; T = 1 reads no stride, so strides that are no multiple of 16 (obs) or 8 (actions) bytes pass
    act1 = torch.zeros(n * 6 + 1, device="cuda").as_strided((1, n, 6), (n * 6 + 1, 6, 1))      # view() would reset stride(0)
    obs1 = torch.zeros(n * 137 + 1, device="cuda").as_strided((1, n, 137), (n * 137 + 1, 137, 1))
    rew1, flg1 = torch.zeros((1, n), device="cuda"), torch.zeros((1, n), dtype=torch.uint8, device="cuda")
    launches = a.launch_count
    _cabi.check(a._lib.pnr_step_many(a._h, 0, act1.data_ptr(), 1, obs1.data_ptr(), 1, rew1.data_ptr(), flg1.data_ptr(),
                                     a._stream()), "pnr_step_many")
    assert a.launch_count == launches
    act1[0] = uniform_actions(a, g, 1)[0]
    assert act1.stride(0) * 4 % 8 and obs1.stride(0) * 4 % 16
    a.step_many(act1, obs1, rew1, flg1)
    assert a.launch_count == launches + 1
    o, r, f = b.step_tensor(act1[0])
    assert torch.equal(f, flg1[0]) and torch.equal(r, rew1[0]) and torch.equal(o, obs1[0])
    sa, sb = a.state(), b.state()
    assert all(torch.equal(sa[k], sb[k]) for k in sa)
    assert a.episode_stats() == b.episode_stats()
    a.close(); b.close()


def test_graph_replays_draw_fresh_reset_states():
    """The host call counter that keys the Philox reset draws is a kernel argument, frozen at capture time; the graph
    advances a device-side counter instead (pnr_tick_advance), so an env that restarts in replay k does not restart
    from the state it restarted from in replay k-1.  Checkpoints fold the device-side part into the counter."""
    from pioneer_b200 import BatchConfig, BatchedPioneerEnv
    n, T = 512, 2
    env = BatchedPioneerEnv(n, seed=8, batch_config=BatchConfig(max_episode_steps=1))     # every step ends an episode
    actions = torch.zeros((T, n, 6), device="cuda")
    obs = torch.zeros((T, n, 137), device="cuda")
    rew = torch.zeros((T, n), device="cuda")
    flg = torch.zeros((T, n), dtype=torch.uint8, device="cuda")
    graph = env.capture_rollout(actions, obs, rew, flg)
    tick0 = env.state_dict()["tick"]
    graph.replay(); torch.cuda.synchronize()
    first = env.state()["r"].clone()
    graph.replay(); torch.cuda.synchronize()
    second = env.state()["r"].clone()
    assert (flg & 1).all()
    assert not torch.equal(first, second) and (first != second).any(dim=1).float().mean() > 0.99
    assert env.state_dict()["tick"] == tick0 + 2 * T
    env.load_state_dict(env.state_dict())      # folds the device-side part into the host counter
    assert env.state_dict()["tick"] == tick0 + 2 * T
    env.close()


def test_scene_mirrors_answer_from_device_state():
    from pioneer_b200.envs.pioneer import PioneerKinematicEnv
    env = PioneerKinematicEnv()
    env.reset_world(joint_positions=np.zeros(6, np.float32), target_position=(20.0, 0.0, 4.0))
    np.testing.assert_allclose(env.scene.items_by_name["robot:pointer"].pose().xyz, (14.6, 1.0, 15.9), atol=1e-5)
    np.testing.assert_allclose(env.scene.items_by_name["target"].pose().xyz, (20.0, 0.0, 4.0))
    assert [j.position() for j in env.scene.joints] == [0.0] * 6 and env.scene.joints[0].velocity() == 0.0
    env.scene.joints[1].reset_state(0.5)
    np.testing.assert_allclose(env.joint_positions(), [0, 0.5, 0, 0, 0, 0])
    env.close()


def test_rollout_worker_collects_fragments_on_the_device():
    from pioneer_b200 import BatchConfig, BatchedPioneerEnv
    from pioneer_b200.rollout import RolloutWorker
    n, T = 512, 6
    env = BatchedPioneerEnv(n, seed=3, batch_config=BatchConfig(max_episode_steps=10))
    w = RolloutWorker(env, fragment_length=T, policy_dtype=torch.float32)
    for it in range(4):
        b = w.collect()
        assert b["obs"].shape == (T, n, 137) and b["actions"].shape == (T, n, 6) and b["reward"].shape == (T, n)
        a_max = torch.as_tensor(env.a_max).cuda()
        assert (b["actions"].abs() <= a_max).all() and torch.isfinite(b["obs"]).all() and torch.isfinite(b["logp"]).all()
        assert float(b["obs"].abs().max()) <= 10.0                      # normalised + clipped
        s = w.sync()
    # 24 steps with TimeLimit 10: every env finished 2 episodes, the last sync window saw the second batch; the filter saw
    # the reset observations, every step's observation and the 2 fresh observations that replaced terminal rows
    assert s["env_steps"] == n * T and w.filter.n == n * (4 * T + 1 + 2)
    assert env.episode_stats()["episodes"] == 0 and s["episodes_total"] == n
    # fragments chain: the first observation of a fragment is the last of the previous one
    last = w.obs[T].clone()
    b = w.collect()
    assert torch.equal(b["obs"][0], last)
    env.close()


def test_checkpoint_resume_is_bit_identical(tmp_path):
    from pioneer_b200 import BatchConfig, BatchedPioneerEnv
    n = 700
    g = torch.Generator(device="cuda").manual_seed(2)
    env = BatchedPioneerEnv(n, seed=6, batch_config=BatchConfig(max_episode_steps=4))
    acts = (torch.rand((12, n, 6), device="cuda", generator=g) * 2 - 1) * 60
    for t in range(5):
        env.step_tensor(acts[t])
    torch.save(env.state_dict(), tmp_path / "env.pt")
    want = [tuple(x.clone() for x in env.step_tensor(acts[t])) for t in range(5, 12)]
    stats_want = env.episode_stats()
    # a fresh env (different seed, different history) continues from the checkpoint
    other = BatchedPioneerEnv(n, seed=99, batch_config=BatchConfig(max_episode_steps=4))
    other.step_tensor(acts[0])
    other.load_state_dict(torch.load(tmp_path / "env.pt"))
    for k, t in enumerate(range(5, 12)):
        o, r, f = other.step_tensor(acts[t])
        assert torch.equal(o, want[k][0]) and torch.equal(r, want[k][1]) and torch.equal(f, want[k][2]), t
    assert other.episode_stats() == stats_want            # the whole statistics window travels with the checkpoint
    env.close(); other.close()


def test_facade_pickles_as_constructor_arguments():
    import pickle
    from pioneer_b200.envs.pioneer import PioneerKinematicConfig, PioneerKinematicEnv
    env = PioneerKinematicEnv(pioneer_config=PioneerKinematicConfig(award_done=7.5))
    clone = pickle.loads(pickle.dumps(env))                       # EzPickle semantics: re-constructed, not copied
    assert isinstance(clone, PioneerKinematicEnv) and clone.config.award_done == 7.5
    assert clone.reset().shape == (137,)
    env.close(); clone.close()


def test_rollout_worker_replays_fragments_from_a_cuda_graph():
    """cuda_graph=True: policy, sampling and env steps of a fragment are captured once and replayed; the statistics,
    the fused normaliser and the reset counter keep advancing on the device."""
    from pioneer_b200 import BatchConfig, BatchedPioneerEnv
    from pioneer_b200.rollout import RolloutWorker
    n, T = 512, 5
    env = BatchedPioneerEnv(n, seed=3, batch_config=BatchConfig(max_episode_steps=4))
    w = RolloutWorker(env, fragment_length=T, policy_dtype=torch.float32, cuda_graph=True)
    a_max = torch.as_tensor(env.a_max).cuda()
    w.collect()                                # warm-up fragment + capture + first replay
    episodes = w.sync()["episodes_total"]
    seen = []
    for it in range(3):
        last = w.obs[T].clone()
        b = w.collect()
        assert torch.equal(b["obs"][0], last)                          # fragments chain
        assert (b["actions"].abs() <= a_max).all() and torch.isfinite(b["obs"]).all() and torch.isfinite(b["logp"]).all()
        assert float(b["obs"].abs().max()) <= 10.0
        s = w.sync()
        assert s["env_steps"] == n * T and s["episodes_total"] >= n    # TimeLimit 4 < T: every env finished an episode
        episodes += s["episodes_total"]
        seen.append((b["actions"].clone(), b["obs"][-1].clone()))
    assert not torch.equal(seen[0][0], seen[1][0])                     # fresh noise on every replay
    assert not torch.equal(seen[1][1], seen[2][1])
    # reset obs + warm-up + capture replay + 3 fragments, plus one fresh observation per finished episode (observe_done)
    assert w.filter.n == n * (1 + 5 * T) + episodes
    env.close()


def test_policy_input_after_done_is_the_reset_observation():
    """ADVICE r1: RLlib's sampler feeds the policy the RESET observation after a done (bullet_env.py:187-197).  The worker
    keeps terminal-observation stepping and patches the finished rows (pnr_observe_done); `episode_start` marks them."""
    from pioneer_b200 import BatchConfig, BatchedPioneerEnv
    from pioneer_b200.rollout import RolloutWorker
    n, T, limit = 300, 7, 3                                            # n not a multiple of 4: padded observation rows
    env = BatchedPioneerEnv(n, seed=5, batch_config=BatchConfig(max_episode_steps=limit))
    w = RolloutWorker(env, fragment_length=T, policy_dtype=torch.float32, use_filter=False, keep_terminal_obs=True)
    b = w.collect()
    done = b["done"]
    assert done[limit - 1].all() and done[2 * limit - 1].all() and not done[0].any()
    assert torch.equal(b["episode_start"][1:], done[:-1]) and not b["episode_start"][0].any()
    t = limit - 1
    fresh = b["next_obs"][t]                                           # = the policy input of step t + 1
    assert torch.equal(fresh, b["obs"][t + 1])
    assert (fresh[:, 90:96] == 0).all() and (fresh[:, 108:114] == 0).all() and (fresh[:, 136] == 0).all()   # a new episode
    term = b["terminal_obs"][t]
    assert (term[:, 136] > 0).all() and not torch.equal(term[:, 0:6], fresh[:, 0:6])
    # the reward of the first step of the new episode carries the whole potential -- paired with the fresh observation
    assert torch.allclose(b["reward"][t + 1], b["obs"][t + 2][:, 136] - 0.01, atol=1e-4)
    # the state the env continues from is the one the policy saw
    w2_obs = env.observe()
    assert torch.equal(w2_obs[:, 129:132], b["next_obs"][-1][:, 129:132])
    b2 = w.collect()
    assert torch.equal(b2["episode_start"][0], done[-1])
    env.close()


def test_compact_host_layout_and_async_double_buffering():
    """pnr_step_host_begin / _end: PNR_HOST_COMPACT rows (101 columns) re-expand to the 137-column rows bit for bit, and two
    steps in flight deliver the same results as synchronous stepping."""
    from pioneer_b200 import BatchConfig, BatchedPioneerEnv
    n, steps = 5000, 9
    a = BatchedPioneerEnv(n, seed=2, batch_config=BatchConfig(max_episode_steps=4))
    b = BatchedPioneerEnv(n, seed=2, batch_config=BatchConfig(max_episode_steps=4))
    rng = np.random.default_rng(0)
    acts = [torch.as_tensor((rng.uniform(-1, 1, size=(n, 6)) * a.a_max).astype(np.float32)).pin_memory() for _ in range(steps)]
    want = []
    for k in range(steps):
        o, r, f = a.step_host(acts[k])
        want.append((o.copy(), r.copy(), f.copy()))
    const = b.obs_constants()
    assert np.array_equal(const, want[0][0][0, 18:54])
    got = []
    b.step_host_begin(acts[0], compact=True)
    for k in range(steps):
        if k + 1 < steps:
            b.step_host_begin(acts[k + 1], compact=(k % 2 == 1))      # two in flight; layouts may alternate
        o, r, f = b.step_host_end()
        full = b.expand_compact(o) if o.shape[1] == 101 else o
        got.append((full.copy(), r.copy(), f.copy()))
    for k in range(steps):
        assert np.array_equal(got[k][0], want[k][0]) and np.array_equal(got[k][1], want[k][1])
        assert np.array_equal(got[k][2], want[k][2])
    with pytest.raises(Exception):
        b.step_host_end()                                              # nothing in flight
    b.step_host_begin(acts[0]); b.step_host_begin(acts[1])
    with pytest.raises(Exception):
        b.step_host_begin(acts[2])                                     # a third step would overwrite a buffer in flight
    b.step_host_end(); b.step_host_end()
    a.close(); b.close()


def test_misaligned_buffers_are_rejected_not_faulted():
    from pioneer_b200 import BatchedPioneerEnv, _cabi
    n = 37
    env = BatchedPioneerEnv(n, seed=1)
    raw = torch.zeros(n * 137 + 8, device="cuda")
    mis = raw[1:1 + n * 137].view(n, 137)                              # 4 bytes off a 16-byte boundary
    lib, h, s = env._lib, env._h, env._stream()
    assert lib.pnr_reset(h, None, n, None, None, mis.data_ptr(), s) != 0
    assert lib.pnr_observe(h, None, n, mis.data_ptr(), s) != 0
    act = torch.zeros((n, 6), device="cuda")
    rew, flg = torch.zeros(n, device="cuda"), torch.zeros(n, dtype=torch.uint8, device="cuda")
    assert lib.pnr_step(h, act.data_ptr(), mis.data_ptr(), rew.data_ptr(), flg.data_ptr(), s) != 0
    torch.cuda.synchronize()                                            # no sticky fault: the device still works
    assert env.observe().shape == (n, 137)
    env.close()


def test_filter_outlives_nothing_and_is_the_identity_before_its_first_sync():
    from pioneer_b200 import BatchedPioneerEnv, _cabi
    from pioneer_b200.obs_filter import MeanStdObsFilter
    env = BatchedPioneerEnv(64, seed=1)
    f = MeanStdObsFilter(env)
    x = torch.randn((64, 137), device="cuda") * 3
    y = f(x.clone())
    assert torch.equal(y, x.clamp(-10, 10))                             # count == 0: identity (then clipped)
    f.sync()
    z = f(x.clone(), update=False)
    assert float(z.mean().abs()) < 0.2 and abs(float(z.std()) - 1.0) < 0.2
    sd = env.state_dict()
    assert sd["obs_filter"]["count"] == 64
    env.close()
    with pytest.raises(_cabi.PioneerB200Error):
        f(x)

