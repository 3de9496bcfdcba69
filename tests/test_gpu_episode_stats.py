"""Episode statistics and the cross-rank statistics exchange against float64 references.

The step kernels add exactly the float32 reward they emit to an env's return (__fadd_rn), so a float32 replay of the
emitted rewards and flags gives every episode's return bit for bit.  From those episodes the reference builds the
eight-number window exactly (math.fsum); the kernels' window must then agree:

  * episodes, sum of lengths, reached_target and env_steps exactly, max and min return bit for bit;
  * the sum of returns within 6u * sum |ret| and the sum of squared returns within 7u * sum ret^2 (u = 2^-24): a warp
    adds its finished episodes in float32 with a depth-5 butterfly before one float64 atomic, and squares in float32.

Covered: K1 (both arithmetic and observation modes, single steps and fragments, obstacles with a random box), K2 (PD,
Bullet-like and torque control), a graph-replayed fragment, pnr_step_host, windows cleared mid-episode, set_state and
reset(indices) mid-run; RolloutWorker.sync()'s summary; pnr_stats_merge_device and pnr_iteration_sync against a left fold
in rank order; the observation filter's exchange at every demean / destd setting against one BatchSyncFilter
(oracle/filter_oracle.py) fed every rank's rows.

The reward here has a larger step penalty (5 instead of 0.01) and a done distance of 5: with the reference's values every
episode return of a random policy is positive (the first reward of an episode is the whole starting potential), and a
square taken as ret * |ret| would go unnoticed."""
import ctypes as C
import json
import math

import numpy as np
import pytest

torch = pytest.importorskip("torch")

U = 2.0 ** -24
REWARD = dict(penalty_step=5.0, done_distance=5.0)
LIMIT = 7
FIELDS = ("episodes", "sum_return", "sum_length", "sum_return_sq", "max_return", "min_return", "env_steps",
          "reached_target")


# ---------------------------------------------------------------------------------------------
# the per-episode reference
# ---------------------------------------------------------------------------------------------
def _host(x, dtype):
    if isinstance(x, torch.Tensor):
        x = x.cpu().numpy()
    return np.asarray(x).astype(dtype)


class EpisodeReference:
    """Replays emitted rewards [T, n] and flags [T, n] of auto-resetting envs from the return and elapsed steps at the
    window start: ret = float32(ret + rew), t += 1; a done records (ret, t, reached = not TRUNCATED) and restarts the
    episode.  Episodes still running are carried over a clear()."""

    def __init__(self, ep_return, t):
        self.ret = _host(ep_return, np.float32).copy()
        self.t = _host(t, np.int64).copy()
        self.clear()

    def clear(self):
        self.returns, self.lengths, self.reached, self.env_steps = [], [], [], 0

    def step(self, reward, flags):
        n = self.ret.size
        for rew, fl in zip(_host(reward, np.float32).reshape(-1, n), _host(flags, np.uint8).reshape(-1, n)):
            self.ret += rew                                     # float32 + float32, rounded to float32
            self.t += 1
            done = (fl & 1) != 0
            self.returns.append(self.ret[done].copy())
            self.lengths.append(self.t[done].copy())
            self.reached.append((fl[done] & 2) == 0)
            self.ret[done] = 0.0
            self.t[done] = 0
            self.env_steps += n

    def restart(self, idx, ep_return=0.0, t=0):
        """set_state(ep_return=..., t=...) or reset(indices): the envs' running episodes are replaced, never recorded."""
        self.ret[idx] = ep_return
        self.t[idx] = t


def reference_window(refs):
    """The merged window of the references (ranks in order): the eight fields, and sum |ret|."""
    def cat(lists, dtype):
        return np.concatenate([x for r in refs for x in lists(r)] or [np.zeros(0, dtype)]).astype(dtype)
    ret = cat(lambda r: r.returns, np.float64)
    w = dict(episodes=float(ret.size), sum_return=math.fsum(ret), sum_length=float(cat(lambda r: r.lengths, np.int64).sum()),
             sum_return_sq=math.fsum(ret * ret),             # a float32 squared is exact in float64
             max_return=float(ret.max()) if ret.size else -math.inf, min_return=float(ret.min()) if ret.size else math.inf,
             env_steps=float(sum(r.env_steps for r in refs)), reached_target=float(cat(lambda r: r.reached, bool).sum()))
    return w, math.fsum(np.abs(ret))


def _bits(x):
    return np.float64(x).view(np.int64)


def assert_window(got, refs, signs=True):
    """`got`: the kernels' window (dict of FIELDS, or the packed float64[8])."""
    if not isinstance(got, dict):
        got = dict(zip(FIELDS, _host(got, np.float64)[:8].tolist()))
    want, abs_sum = reference_window(refs)
    if signs:
        assert want["min_return"] < 0.0 < want["max_return"], "the window must hold negative and positive returns"
    for key in ("episodes", "sum_length", "reached_target", "env_steps"):
        assert got[key] == want[key], (key, got[key], want[key])
    for key in ("max_return", "min_return"):
        assert _bits(got[key]) == _bits(want[key]), (key, got[key], want[key])
    d1 = abs(got["sum_return"] - want["sum_return"])
    assert d1 <= 6 * U * abs_sum, ("sum_return", got["sum_return"], want["sum_return"], d1 / max(abs_sum, 1e-300))
    d2 = abs(got["sum_return_sq"] - want["sum_return_sq"])
    assert d2 <= 7 * U * want["sum_return_sq"], ("sum_return_sq", got["sum_return_sq"], want["sum_return_sq"])
    return want


def test_episode_reference_known_answer():
    """Three envs, four steps: two episodes end reached, two by TimeLimit; float32 accumulation (2^24 + 1 + 1 stays 2^24)."""
    ref = EpisodeReference(np.array([0.5, 2.0 ** 24, -1.0], np.float32), np.array([0, 5, 2]))
    reward = np.array([[1.0, 1.0, 0.25], [-3.0, 1.0, 0.5], [2.0, 0.5, 4.0], [0.75, -2.0, 1.0]], np.float32)
    flags = np.array([[0, 0, 0], [1, 3, 0], [0, 0, 3], [1, 0, 0]], np.uint8)
    ref.step(reward[:1], flags[:1])                         # one step, then a fragment of three
    ref.step(reward[1:], flags[1:])
    want, abs_sum = reference_window([ref])
    assert want == dict(episodes=4.0, sum_return=-1.5 + 2.0 ** 24 + 3.75 + 2.75, sum_length=2.0 + 7 + 5 + 2,
                        sum_return_sq=2.25 + 2.0 ** 48 + 14.0625 + 7.5625, max_return=2.0 ** 24, min_return=-1.5,
                        env_steps=12.0, reached_target=2.0)
    assert abs_sum == 1.5 + 2.0 ** 24 + 3.75 + 2.75
    assert ref.ret.tolist() == [0.0, -1.5, 1.0] and ref.t.tolist() == [0, 2, 1]
    ref.clear()
    ref.restart([1], 2.5, 3)
    ref.step(np.array([[1.0, 0.5, -4.0]], np.float32), np.array([[0, 1, 0]], np.uint8))
    want, _ = reference_window([ref])
    assert want["episodes"] == 1 and want["sum_return"] == 3.0 and want["sum_length"] == 4 and want["reached_target"] == 1
    ref.clear()
    empty, abs_sum = reference_window([ref, ref])           # nothing ended: the cleared window's extrema
    assert empty == dict(episodes=0.0, sum_return=0.0, sum_length=0.0, sum_return_sq=0.0, max_return=-math.inf,
                         min_return=math.inf, env_steps=0.0, reached_target=0.0) and abs_sum == 0.0
    assert_window(empty, [ref], signs=False)


# ---------------------------------------------------------------------------------------------
# one handle's window
# ---------------------------------------------------------------------------------------------
def _kinematic(n, seed=0, env_id_base=0, **fields):
    from tests._gpu import kinematic_env
    return kinematic_env(n, seed=seed, env_id_base=env_id_base, **{"max_episode_steps": LIMIT, **REWARD, **fields})


def _dynamic(n, control, seed=0):
    from pioneer_b200 import BatchConfig, BatchedPioneerEnv, PioneerKinematicConfig, SimulationConfig
    from tests._gpu import CONTROL
    fields = dict(CONTROL[control])
    gravity = fields.pop("gravity", 0.0)
    return BatchedPioneerEnv(n, seed=seed, pioneer_config=PioneerKinematicConfig(**REWARD),
                             simulation_config=SimulationConfig(gravity=gravity),
                             batch_config=BatchConfig(mode="dynamic", max_episode_steps=LIMIT, **fields))


def _driver(env, launch, T, gen):
    """advance(): the next T steps of `env` under uniform actions, launched as `launch` ("step": one pnr_step per step,
    "fragment": one pnr_step_many, "graph": a captured fragment replayed, "host": pnr_step_host per step); returns the
    emitted reward [T, n] and flags [T, n] on the host."""
    from tests._gpu import fragment_buffers, uniform_actions
    n = env.n_envs
    if launch in ("step", "host"):
        def advance():
            act = uniform_actions(env, gen, T)
            rew, flg = np.empty((T, n), np.float32), np.empty((T, n), np.uint8)
            for t in range(T):
                if launch == "step":
                    _, r, f = env.step_tensor(act[t])
                    rew[t], flg[t] = r.cpu().numpy(), f.cpu().numpy()
                else:
                    _, r, f = env.step_host(act[t].cpu().numpy())
                    rew[t], flg[t] = r, f
            return rew, flg
        return advance
    act = uniform_actions(env, gen, T)
    obs, rew, flg = fragment_buffers(T, n)
    graph = env.capture_rollout(act, obs, rew, flg) if launch == "graph" else None   # capturing runs one step

    def advance():
        act.copy_(uniform_actions(env, gen, T))
        if graph is None:
            env.step_many(act, obs, rew, flg)
        else:
            graph.replay()
        return rew.cpu().numpy(), flg.cpu().numpy()
    return advance


def window_rounds(env, launch, T, *, chunks, rounds=3, seed=0):
    """`rounds` windows of `chunks` x T steps, each compared with the reference and cleared, so episodes straddle the
    clears.  Mid-way through round 1 every env's return and elapsed steps are replaced (set_state); mid-way through round 2
    a fifth of the envs restart mid-episode (reset(indices)), and their partial episodes are never counted."""
    n = env.n_envs
    rng = np.random.default_rng(seed)
    advance = _driver(env, launch, T, torch.Generator(device="cuda").manual_seed(seed))
    env.episode_stats(clear=True)
    s = env.state()
    ref = EpisodeReference(s["ep_return"], s["t"])
    for k in range(rounds):
        for c in range(chunks):
            if c == chunks // 2 and k == 1:
                ep = rng.uniform(-40.0, 40.0, n).astype(np.float32)
                t = rng.integers(0, LIMIT, n).astype(np.int32)
                env.set_state(ep_return=ep, t=t)
                ref.restart(slice(None), ep, t)
            if c == chunks // 2 and k == 2:
                idx = np.sort(rng.choice(n, size=max(1, n // 5), replace=False))
                env.reset(idx)
                ref.restart(idx)
            ref.step(*advance())
        assert_window(env.episode_stats(clear=True), [ref])
        ref.clear()
    s = env.state()                                         # the episodes still running at the end, too
    assert np.array_equal(s["ep_return"].cpu().numpy(), ref.ret) and np.array_equal(s["t"].cpu().numpy(), ref.t)
    env.close()


SHAPES = [77, 4096 + 37, 65536]


@pytest.mark.gpu
@pytest.mark.parametrize("n", SHAPES)
@pytest.mark.parametrize("T", [1, 8, 17])
@pytest.mark.parametrize("arith,obs_mode", [("f32", "terminal"), ("f32", "autoreset"), ("legacy64", "terminal"),
                                            ("legacy64", "autoreset")])
def test_k1_window_equals_the_episode_reference(arith, obs_mode, T, n):
    """T = 1: single steps (8 per chunk); T = 8 / 17: pnr_step_many fragments."""
    env = _kinematic(n, seed=T + n, arith=arith, obs_mode=obs_mode)
    if T == 1:
        window_rounds(env, "step", 8, chunks=2, seed=n)
    else:
        window_rounds(env, "fragment", T, chunks=2, seed=n)


@pytest.mark.gpu
@pytest.mark.parametrize("launch,T", [("step", 8), ("fragment", 8), ("fragment", 17)])
def test_k1_obstacles_window_equals_the_episode_reference(launch, T):
    """The obstacle variant adds the contact penalty, the return and the statistics behind the tile's DONE barrier."""
    window_rounds(_kinematic(4096 + 37, seed=5, obstacles=True), launch, T, chunks=2, seed=5)


@pytest.mark.gpu
@pytest.mark.parametrize("launch", ["step", "fragment"])
@pytest.mark.parametrize("control", ["pd", "bullet", "torque"])
def test_k2_window_equals_the_episode_reference(control, launch):
    window_rounds(_dynamic(4096 + 37, control, seed=7), launch, 8, chunks=2, seed=7)


@pytest.mark.gpu
def test_graph_replayed_fragments_window_equals_the_episode_reference():
    window_rounds(_kinematic(4096 + 37, seed=11), "graph", 8, chunks=2, seed=11)


@pytest.mark.gpu
def test_step_host_window_equals_the_episode_reference():
    window_rounds(_kinematic(1000, seed=13), "host", 8, chunks=2, seed=13)


# ---------------------------------------------------------------------------------------------
# RolloutWorker.sync(): the summary of the window
# ---------------------------------------------------------------------------------------------
def assert_summary(got, refs):
    """summarize() of the kernels' window against the reference: the bars of assert_window, carried through the mean and
    the standard deviation (plus float64 rounding of summarize itself on either side)."""
    want, abs_sum = reference_window(refs)
    n = want["episodes"]
    assert want["min_return"] < 0.0 < want["max_return"], "the window must hold negative and positive returns"
    assert got["episodes_total"] == n and got["env_steps"] == want["env_steps"]
    assert got["reached_target"] == want["reached_target"]
    assert _bits(got["episode_reward_max"]) == _bits(want["max_return"])
    assert _bits(got["episode_reward_min"]) == _bits(want["min_return"])
    assert got["episode_len_mean"] == want["sum_length"] / n
    e1, e2 = 6 * U * abs_sum / n, 7 * U * want["sum_return_sq"] / n
    mean = want["sum_return"] / n
    assert abs(got["episode_reward_mean"] - mean) <= e1 + 2.0 ** -52 * abs(mean), (got["episode_reward_mean"], mean)
    mean_sq = want["sum_return_sq"] / n
    var = max(mean_sq - mean * mean, 0.0)
    dvar = e2 + 2 * abs(mean) * e1 + e1 * e1 + 2.0 ** -50 * (mean_sq + mean * mean)
    std = math.sqrt(var)
    bound = min(math.sqrt(dvar), dvar / std) if std > 0.0 else math.sqrt(dvar)   # |sqrt a - sqrt b| <= |a - b| / sqrt b
    assert abs(got["episode_reward_std"] - std) <= bound, (got["episode_reward_std"], std, bound)


@pytest.mark.gpu
@pytest.mark.parametrize("cuda_graph", [False, True])
def test_rollout_worker_summary_equals_the_episode_reference(cuda_graph):
    """512 + 3 envs, TimeLimit 4, fragments of 8 (fused filter, terminal observations, in-kernel auto-reset); the
    reference replays collect()'s reward / done / truncated.  A sync with no step since the last one reports None for
    every per-episode number, never NaN."""
    from pioneer_b200.rollout import RolloutWorker
    env = _kinematic(512 + 3, seed=17, max_episode_steps=4)
    w = RolloutWorker(env, fragment_length=8, seed=17, cuda_graph=cuda_graph)
    w.collect()
    w.sync()                                                # the window restarts here
    s = env.state()
    ref = EpisodeReference(s["ep_return"], s["t"])
    for it in range(3):
        for _ in range(2):
            out = w.collect()
            ref.step(out["reward"], out["done"].to(torch.uint8) | (out["truncated"].to(torch.uint8) << 1))
        assert_summary(w.sync(), [ref])
        ref.clear()
    empty = w.sync()
    assert empty["episodes_total"] == 0.0 and empty["env_steps"] == 0.0 and empty["reached_target"] == 0.0
    for key in ("episode_reward_mean", "episode_reward_std", "episode_reward_max", "episode_reward_min",
                "episode_len_mean"):
        assert empty[key] is None, key
    json.dumps(empty, allow_nan=False)
    env.close()


# ---------------------------------------------------------------------------------------------
# the cross-rank merge
# ---------------------------------------------------------------------------------------------
def rank_fold(rows):
    """The windows [world, len] combined in rank order: a left fold, SUM everywhere except MAX at 4 and MIN at 5."""
    rows = np.asarray(rows, np.float64)
    acc = rows[0].copy()
    for x in rows[1:]:
        nxt = acc + x
        nxt[4], nxt[5] = max(acc[4], x[4]), min(acc[5], x[5])
        acc = nxt
    return acc


@pytest.mark.gpu
@pytest.mark.parametrize("extra", [0, 275])
def test_stats_merge_device_is_the_rank_order_fold(extra):
    """Synthetic windows of 1 - 16 ranks (8 statistics, or 8 + the filter's 275 sums): mixed signs over nine decades, so
    that the summation order shows in the last bits; empty windows (+-inf extrema, zero sums), +inf in a sum, ties."""
    from pioneer_b200 import _cabi as c
    assert extra in (0, c.PNR_FILTER_DELTA_LEN)
    lib = c.load()
    length = 8 + extra
    rng = np.random.default_rng(extra)
    out = torch.empty(length, dtype=torch.float64, device="cuda")
    for world in range(1, 17):
        rows = rng.normal(size=(world, length)) * 10.0 ** rng.integers(-4, 5, size=(world, length))
        rows[:, 4] = rng.choice([-2.5, 1.0, 7.25], size=world)           # ties among the extrema
        rows[:, 5] = rng.choice([-2.5, 1.0, 7.25], size=world)
        if world > 1:
            empty = rng.integers(world)
            rows[empty, :4] = 0.0
            rows[empty, 4:6] = (-math.inf, math.inf)
            rows[rng.integers(world), 4] = math.inf
            rows[rng.integers(world), 5] = -math.inf
        if world == 7:
            rows[3, 2] = math.inf
        gathered = torch.as_tensor(rows).cuda()
        out.fill_(math.nan)
        c.check(lib.pnr_stats_merge_device(gathered.data_ptr(), world, length, out.data_ptr(), None))
        torch.cuda.synchronize()
        want = rank_fold(rows)
        assert np.array_equal(out.cpu().numpy().view(np.int64), want.view(np.int64)), world
        if world > 2:                                        # the fold is order-sensitive here: a reordering would show
            assert not np.array_equal(rank_fold(rows[::-1]).view(np.int64), want.view(np.int64))
    rows = torch.zeros((2, 8), dtype=torch.float64, device="cuda")
    assert lib.pnr_stats_merge_device(rows.data_ptr(), 0, 8, out.data_ptr(), None) != 0
    assert lib.pnr_stats_merge_device(rows.data_ptr(), 2, 7, out.data_ptr(), None) != 0


def _sync_all(envs, with_filter, outs, streams, rotate):
    """One pnr_iteration_sync per rank (clearing the windows), launched in a rotating order on concurrent streams."""
    from pioneer_b200 import _cabi as c
    world = len(envs)
    torch.cuda.synchronize()
    for r in range(world):
        q = (r + rotate) % world
        with torch.cuda.stream(streams[q]):
            c.check(envs[q]._lib.pnr_iteration_sync(envs[q]._h, int(with_filter), 1, outs[q].data_ptr(), 5000,
                                                     streams[q].cuda_stream))
    torch.cuda.synchronize()
    for e in envs:
        flag = C.c_int(-1)
        c.check(e._lib.pnr_sync_status(e._h, C.byref(flag)))
        assert flag.value == 0                              # no rank gave up waiting


@pytest.mark.gpu
@pytest.mark.parametrize("world", [1, 2, 3, 4])
def test_iteration_sync_is_the_rank_order_fold_of_the_windows(world):
    """Handles on one GPU play the ranks (as in test_gpu_sync.py).  Every rank's output is bit for bit the rank-order fold
    of the windows each rank reported (pnr_stats, no clear) just before the exchange, and within the bars of the merged
    per-episode references.  In round 1 the last rank takes no step: its window is empty (at world 1 the merged one is)."""
    from tests._gpu import fragment_buffers, uniform_actions
    from tests.test_gpu_sync import _connect
    n, T = 1000, 6
    envs = [_kinematic(n, seed=19, env_id_base=r * n) for r in range(world)]
    if world > 1:
        _connect(envs)
    gen = torch.Generator(device="cuda").manual_seed(19)
    bufs = fragment_buffers(T, n)
    refs = []
    for e in envs:
        e.episode_stats(clear=True)
        s = e.state()
        refs.append(EpisodeReference(s["ep_return"], s["t"]))
    outs = [torch.zeros(8, dtype=torch.float64, device="cuda") for _ in range(world)]
    streams = [torch.cuda.Stream() for _ in range(world)]
    for k in range(4):
        for r, (e, ref) in enumerate(zip(envs, refs)):
            if k == 1 and r == world - 1:
                continue
            for _ in range(2 + (k + r) % 2):
                e.step_many(uniform_actions(e, gen, T), *bufs)
                ref.step(bufs[1], bufs[2])
        snapshots = [[e.episode_stats()[f] for f in FIELDS] for e in envs]
        _sync_all(envs, False, outs, streams, k)
        want = rank_fold(snapshots)
        for r in range(world):
            assert np.array_equal(outs[r].cpu().numpy().view(np.int64), want.view(np.int64)), (k, r)
        if k == 1:
            assert snapshots[-1][0] == 0.0 and snapshots[-1][4] == -math.inf and snapshots[-1][5] == math.inf
        assert_window(outs[0], refs, signs=not (k == 1 and world == 1))
        for e, ref in zip(envs, refs):
            assert e.episode_stats()["env_steps"] == 0.0                    # every window was cleared
            ref.clear()
    for e in envs:
        e.close()


# ---------------------------------------------------------------------------------------------
# the observation filter across ranks
# ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("demean,destd", [(True, True), (False, True), (True, False)])
@pytest.mark.parametrize("world", [1, 2, 3])
def test_filter_exchange_equals_one_batch_filter_of_all_ranks(world, demean, destd):
    """Ranks push raw observation rows (MeanStdObsFilter.push, 1 - 3 batches of a ragged 333 rows per rank and round) and
    exchange them through pnr_iteration_sync.  The reference is ONE BatchSyncFilter fed every rank's rows in rank order and
    synchronised at the same points.  After each exchange, on every rank: the row count exactly, mean and variance within
    the filter tests' bars, bit-identical statistics on all ranks, and a batch normalised without update within 2e-5."""
    from oracle.filter_oracle import BatchSyncFilter
    from pioneer_b200 import _cabi as c
    from pioneer_b200.obs_filter import MeanStdObsFilter
    from tests._gpu import uniform_actions
    from tests.test_gpu_sync import _connect
    n = 333
    envs = [_kinematic(n, seed=23, env_id_base=r * n) for r in range(world)]
    flts = [MeanStdObsFilter(e, demean=demean, destd=destd) for e in envs]
    if world > 1:
        _connect(envs)
    ora = BatchSyncFilter(c.PNR_OBS_DIM, demean=demean, destd=destd)
    gen = torch.Generator(device="cuda").manual_seed(23)
    outs = [torch.zeros(8 + c.PNR_FILTER_DELTA_LEN, dtype=torch.float64, device="cuda") for _ in range(world)]
    streams = [torch.cuda.Stream() for _ in range(world)]
    for k in range(4):
        for r, (e, f) in enumerate(zip(envs, flts)):
            for _ in range(1 + (k + r) % 3):
                obs, _, _ = e.step_tensor(uniform_actions(e, gen, 1)[0])
                f.push(obs)
                ora(obs.cpu().numpy())
                if r == 0:
                    probe = obs.clone()
        _sync_all(envs, True, outs, streams, k)
        ora.sync()
        stats = [f._get() for f in flts]
        for r, (cnt, mean, var) in enumerate(stats):
            assert cnt == ora.rs.n, (k, r, cnt, ora.rs.n)
            np.testing.assert_allclose(mean, ora.rs.M, rtol=1e-6, atol=1e-6, err_msg=f"round {k} rank {r}")
            np.testing.assert_allclose(var, ora.rs.var, rtol=1e-5, atol=1e-9, err_msg=f"round {k} rank {r}")
            assert np.array_equal(mean, stats[0][1]) and np.array_equal(var, stats[0][2]), (k, r)
            y = flts[r](probe.clone(), update=False)
            np.testing.assert_allclose(y.cpu().numpy(), ora(probe.cpu().numpy(), update=False), rtol=0, atol=2e-5,
                                       err_msg=f"round {k} rank {r}")
        assert torch.equal(outs[0][8:], outs[-1][8:])
    for e in envs:
        e.close()
