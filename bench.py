#!/usr/bin/env python
"""Benchmark of the hot path: env-steps/sec of the batched Pioneer 6-DoF reach env on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--envs-per-gpu E] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

One JSON line on stdout (rank 0).  A "step" is ONE fused-kernel pass of the hot path over the whole
batch of envs with synthetic random actions (BASELINE.json configs[2]: 65,536 envs per GPU, joint limits,
TimeLimit 500, in-kernel auto-reset; weak scaling: every rank owns its own 65,536 envs, no data-path
collective).  See DESIGN.md "Measurement" for what each key means and how the bytes are counted.

`--impl reference` times the reference's CPU path (one env per process on all host cores): the unmodified reference
under PyBullet when pybullet, gym and the reference package are importable, else (PyBullet is not installable offline)
the CPU restatement in oracle/ (the only place besides the `cpu_baseline` leg where this file executes oracle/ code,
and never as the thing shipped).
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "env-steps/sec (6-DoF reach)"
UNIT = "env-steps/s"
DOF, OBS_DIM = 6, 137
# ALGORITHMIC bytes per env-step (SURVEY.md 8(d) D4, DESIGN.md): actions 24 + obs 548 + reward 4 + done 1
# + 23 words of state read and written (92 + 92)
BYTES_IO = 24 + 548 + 4 + 1
BYTES_STATE = 2 * 92
BYTES_PER_ENV_STEP = BYTES_IO + BYTES_STATE          # 761
FRAME_SKIP = 10
FALLBACK_HBM_GBS = 6650.0                            # /opt/skills/guides/B200_PROFILING.md fallback
L2_FLUSH_BYTES = 512 << 20                           # > 4x the 126 MB L2
# Tier-B dynamic kernel, from the committed ncu capture (profiles/r02_step_dynamic_1m.md): 356,253,696 FFMA + 164,900,085
# FMUL + 75,836,005 FADD warp instructions per launch of 2 steps x 32,768 tiles = FFMA 5,436 + FMUL 2,516 + FADD 1,157 thread
# instructions per env-step (10 ABA substeps) = 14,545 flop; FP32 FMA peak measured on this pool's B200 with
# tools/fma_peak.py = 72.6 TFLOP/s (nominal 148 SMs x 128 lanes x 2 x 1.965 GHz = 74.4)
DYN_FLOP_PER_ENV_STEP = 2 * 5436 + 2516 + 1157
DYN_FP_INSTR_PER_ENV_STEP = 5436 + 2516 + 1157
FP32_PEAK_TFLOPS = 72.6
# measured with tools/fp32_forms.py (profiles/r02_fp32_forms.md): a stream of THREE-REGISTER FFMAs issues at 0.711 warp
# instructions per clock per SM sub-partition (operand delivery), two-register FMUL / FADD at 0.976: the FP32 instructions of
# one K2 env-step alone need this many clocks per 32-env tile per sub-partition
DYN_OPERAND_BOUND_CLOCKS = 5436 / 0.711 + (2516 + 1157) / 0.976
SM_SUBPARTITIONS, SM_CLOCK_HZ = 148 * 4, 1.965e9

def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3000)
    ap.add_argument("--warmup", type=int, default=100)
    ap.add_argument("--envs-per-gpu", type=int, default=65536)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-sweep", action="store_true", help="skip the env-count sweep (N=1 only)")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the dynamic-mode / obstacle / rollout-loop records (emitted at every N otherwise)")
    ap.add_argument("--flush", default="write", choices=["write", "write+read", "none"],
                    help="L2 flush between timed steps: 512 MiB memset, optionally followed by a 512 MiB read sweep "
                         "(leaves the L2 full of CLEAN lines instead of dirty ones); 'none' is for profiler launch lists "
                         "only (the number it prints is L2-warm and is not a bench value)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-steps-per-proc", type=int, default=0,
                    help="reference arm: env-steps per process per bench step (0 = sized for ~20 s in total)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned (rank 0: obs, reward, flags) "
                         "as DIR/<name>.npy, so that two builds can be compared output for output on the same inputs")
    return ap.parse_args()


# =================================================================================================
# reference arm / cpu_baseline: the oracle, one env per process on every host core
# =================================================================================================
def _host_cores() -> int:
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def _real_reference_available():
    """BASELINE.md section 4.1 / SURVEY D5: the real thing first.  True when pybullet and gym import and the unmodified
    reference package `pioneer` is importable (installed, on PYTHONPATH, under baseline/_ref, or at $PIONEER_REFERENCE) --
    neither is the case in the build container or on the bench boxes (no wheel, no network), so the port runs there."""
    try:
        import gym  # noqa: F401
        import pybullet  # noqa: F401
    except Exception:  # noqa: BLE001
        return False
    for extra in (os.environ.get("PIONEER_REFERENCE"), os.path.join(ROOT, "baseline", "_ref")):
        if extra and os.path.isdir(extra) and extra not in sys.path:
            sys.path.append(extra)
    try:
        from pioneer.envs.pioneer import PioneerKinematicEnv  # noqa: F401
        return True
    except Exception:  # noqa: BLE001
        return False


def _pybullet_worker(task):
    """One rollout worker of the UNMODIFIED reference: TimeLimit(PioneerKinematicEnv(), 500) exactly as
    pioneer/launch/pioneer_knm_train.py:20-27 builds it, PyBullet DIRECT, random actions, reset on done."""
    proc_id, warm_steps, timed_steps = task
    import numpy as np
    _real_reference_available()
    from gym.wrappers import TimeLimit
    from pioneer.envs.pioneer import PioneerKinematicEnv
    env = TimeLimit(PioneerKinematicEnv(headless=True), max_episode_steps=500)
    env.seed(proc_id)
    env.reset()
    rng = np.random.default_rng(proc_id)
    a_max = env.env.a_max
    actions = (rng.uniform(-1, 1, size=(1024, DOF)) * a_max).astype(np.float32)

    def run(n):
        for t in range(n):
            _, _, done, _ = env.step(actions[t & 1023])
            if done:
                env.reset()

    run(warm_steps)
    t0 = time.perf_counter()
    run(timed_steps)
    return timed_steps, time.perf_counter() - t0


def _cpu_worker(task):
    """One reference-style rollout worker: TimeLimit(PioneerKinematicEnv(), 500) restated by oracle.OracleEnv,
    random actions in [-a_max, a_max], reset on done.  Returns (env_steps, seconds) of the timed part."""
    proc_id, warm_steps, timed_steps = task
    import numpy as np
    from oracle.reach_oracle import OracleChain, OracleEnv
    from pioneer_b200.urdf import flatten_urdf      # host-side table builder only (no CUDA involved)
    env = OracleEnv(OracleChain.from_model(flatten_urdf()), arith="np2", global_env_id=proc_id, seed=0)
    rng = np.random.default_rng(proc_id)
    tick = 0
    env.reset_world(tick=tick)
    actions = (rng.uniform(-1, 1, size=(1024, DOF)) * env.a_max).astype(np.float32)

    def run(n):
        nonlocal tick
        for t in range(n):
            _, _, done, _ = env.step(actions[t & 1023])
            if done:
                tick += 1
                env.reset_world(tick=tick)
                env.observe()

    run(warm_steps)
    t0 = time.perf_counter()
    run(timed_steps)
    return timed_steps, time.perf_counter() - t0


def _c_port_worker(task):
    """The compiled restatement (oracle/reach_oracle.c): 256 envs per process, observations included."""
    proc_id, seconds = task
    import numpy as np
    from oracle.c_oracle import COracleBatch
    from oracle.reach_oracle import OracleChain
    from pioneer_b200.urdf import flatten_urdf
    n = 256
    b = COracleBatch(OracleChain.from_model(flatten_urdf()), n, env_id_base=proc_id * n, seed=0)
    act = (np.random.default_rng(proc_id).uniform(-1, 1, size=(n, DOF)) * b.a_max).astype(np.float32)
    for _ in range(20):
        b.step(act)
    t0, k = time.perf_counter(), 0
    while time.perf_counter() - t0 < seconds:
        for _ in range(20):
            b.step(act)
        k += 20
    return k * n, time.perf_counter() - t0


def run_c_port(seconds: float = 3.0):
    import multiprocessing as mp
    cores = _host_cores()
    with mp.get_context("spawn").Pool(cores) as pool:
        res = pool.map(_c_port_worker, [(i, seconds) for i in range(cores)])
    return sum(r[0] for r in res) / max(r[1] for r in res), cores


def run_cpu_path(steps: int, warmup: int, per_step: int):
    """steps x per_step env-steps on each of P processes.  Returns (value, cores, seconds, per_step)."""
    import multiprocessing as mp
    cores = _host_cores()
    if per_step <= 0:
        # ~1.6k env-steps/s per core for the Python port: aim for ~20 s of timed work per process
        per_step = max(1, min(512, math.ceil(32000 / max(steps, 1))))
    tasks = [(i, warmup * per_step if warmup * per_step < 2000 else 2000, steps * per_step) for i in range(cores)]
    ctx = mp.get_context("spawn")
    real = _real_reference_available()
    with ctx.Pool(cores) as pool:
        res = pool.map(_pybullet_worker if real else _cpu_worker, tasks)
    total = sum(r[0] for r in res)
    slowest = max(r[1] for r in res)
    return total / slowest, cores, slowest, per_step, ("pybullet" if real else "port")


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    value, cores, seconds, per_step, kind = run_cpu_path(args.steps, args.warmup, args.cpu_steps_per_proc)
    try:     # context only: how fast a COMPILED single-thread-per-core port of the same env runs on these cores
        c_value, c_cores = run_c_port()
        c_port = {"value": c_value, "unit": UNIT, "cores": c_cores,
                  "sample": "oracle/reach_oracle.c, 256 envs per process x all cores, ~3 s, observations included"}
    except Exception as exc:  # noqa: BLE001
        c_port = {"value": None, "note": repr(exc)}
    sample = (f"{cores} processes x 1 env each (the reference's rollout-worker layout), {args.steps} steps x "
              f"{per_step} env-steps per process, TimeLimit 500 with resets, random actions; "
              + ("the UNMODIFIED reference env under PyBullet DIRECT" if kind == "pybullet" else
                 "pybullet / gym are not importable here, so this is the Python restatement of the reference env "
                 "(oracle/reach_oracle.py), no PyBullet calls: an upper bound on the real reference's speed"))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * seconds / max(args.steps, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64/f32 (numpy)",
        "data": "synthetic",
        "config": {"workload": "one reach env per host process, random actions, TimeLimit 500",
                   "envs": cores, "env_steps_per_step": cores * per_step},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample,
                         "c_port": c_port},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "substeps_per_sec": value * FRAME_SKIP, "gpu_launches": 0,
    }
    print(json.dumps(_finite(line)), flush=True)


def cpu_baseline_subprocess(seconds_budget: float = 20.0):
    """Run the reference arm in a fresh interpreter (this process holds a CUDA context) and parse its line."""
    steps = 250
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", str(steps), "--warmup", "3",
           "--cpu-steps-per-proc", str(max(1, int(seconds_budget * 1600 / steps)))]
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE")}
    out = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=600)
    for ln in reversed(out.stdout.strip().splitlines()):
        if ln.startswith("{"):
            return json.loads(ln)["cpu_baseline"]
    raise RuntimeError("cpu baseline failed: " + out.stderr[-2000:])


# =================================================================================================
# clocks during the timed region
# =================================================================================================
_REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x10: "sync_boost", 0x20: "sw_thermal_slowdown",
            0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting"}


class ClockSampler(threading.Thread):
    def __init__(self, torch_device_index: int, period_s: float = 0.01):
        super().__init__(daemon=True)
        self.period = period_s
        self.samples, self.bits, self.power = [], 0, []
        self._stop_evt = threading.Event()
        self.ok = False
        self.max_mhz = None
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            self.nv = pynvml
            uuid = str(torch.cuda.get_device_properties(torch_device_index).uuid)
            try:
                self.h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
            except Exception:  # noqa: BLE001
                self.h = pynvml.nvmlDeviceGetHandleByIndex(torch_device_index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception as exc:  # noqa: BLE001
            self.err = repr(exc)

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        while not self._stop_evt.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    self.bits |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:  # noqa: BLE001
                    self.bits |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1e3)
            except Exception:  # noqa: BLE001
                pass
            time.sleep(self.period)

    def finish(self):
        self._stop_evt.set()
        if self.is_alive():
            self.join(timeout=2)
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0,
                    "note": getattr(self, "err", "no samples")}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz,
                "reasons": [name for bit, name in _REASONS.items() if self.bits & bit], "samples": len(s),
                "power_w_max": max(self.power) if self.power else None}


# =================================================================================================
# our arm
# =================================================================================================
FRAGMENT = 8                                         # steps launched back to back between two L2 flushes (a rollout fragment)


def measured_hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    except Exception:  # noqa: BLE001
        return FALLBACK_HBM_GBS, "B200_PROFILING.md fallback (of fallback)"


def ncu_traffic(lib, n):
    """dram__bytes_read.sum + dram__bytes_write.sum per LAUNCH of the step kernel (one launch = one rollout fragment) from an
    `ncu --set full` capture of THIS build: profiles/r02_traffic.json is keyed by the library's source hash
    (pnr_source_hash), so a number captured from other code is never reported -- null instead.
    Returns (bytes per launch, steps per launch in that capture, capture file, source hash)."""
    try:
        import ctypes
        lib.pnr_source_hash.restype = ctypes.c_char_p
        h = lib.pnr_source_hash().decode().split(":", 1)[1]
        with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
            table = json.load(f)
        ent = table.get(h, {}).get(str(n))
        if ent is None:
            return None, None, None, h
        return ent["bytes_per_launch"], ent["steps_per_launch"], ent["capture"], h
    except Exception:  # noqa: BLE001
        return None, None, None, None


def time_fragments(torch, env, actions, obs_ring, reward, flags, steps, warmup, flush, fragment=FRAGMENT):
    """EXACTLY `steps` env steps, launched as rollout fragments of `fragment` steps (pnr_step_many: ONE kernel launch per
    fragment, every CTA / warp runs the fragment's steps on its own tiles; consecutive steps write different slots of the
    observation ring); an untimed L2 flush (512 MiB memset) runs between fragments and every fragment is bracketed by its
    own CUDA-event pair on the launching stream.  Returns (sum of fragment ms, list of (ms, steps) per fragment)."""
    T = min(fragment, obs_ring.shape[0], actions.shape[0])
    done, k = 0, 0
    while done < warmup:
        t = min(T, warmup - done)
        if flush is not None:
            flush()
        env.step_many(actions[:t], obs_ring[:t], reward[:t], flags[:t])
        done += t
    plan, left = [], steps
    while left > 0:
        plan.append(min(T, left))
        left -= plan[-1]
    starts = [torch.cuda.Event(enable_timing=True) for _ in plan]
    stops = [torch.cuda.Event(enable_timing=True) for _ in plan]
    torch.cuda.synchronize()
    launches0 = env.launch_count
    for k, t in enumerate(plan):
        if flush is not None:
            flush()
        starts[k].record()
        env.step_many(actions[:t], obs_ring[:t], reward[:t], flags[:t])
        stops[k].record()
    torch.cuda.synchronize()
    time_fragments.launches = env.launch_count - launches0        # kernels of this library inside the timed region
    per = [(s.elapsed_time(e), t) for s, e, t in zip(starts, stops, plan)]
    return sum(ms for ms, _ in per), per


def time_device_steps(torch, env, actions, obs_ring, reward, flags, steps, warmup, flush):
    """Round-1 method, kept for continuity: every step bracketed by its own event pair, an L2 flush before every step."""
    n_act, n_obs = actions.shape[0], obs_ring.shape[0]
    for k in range(warmup):
        if flush is not None:
            flush()
        env.step_tensor(actions[k % n_act], out=(obs_ring[k % n_obs], reward[0], flags[0]))
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    stops = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    torch.cuda.synchronize()
    for k in range(steps):
        if flush is not None:
            flush()
        starts[k].record()
        env.step_tensor(actions[k % n_act], out=(obs_ring[k % n_obs], reward[0], flags[0]))
        stops[k].record()
    torch.cuda.synchronize()
    per = [s.elapsed_time(e) for s, e in zip(starts, stops)]
    return sum(per), per


def time_graph(torch, env, actions, obs_ring, reward, flags, steps):
    """Back-to-back steps replayed from a CUDA graph of len(obs_ring) steps, no flush: what a device-resident rollout loop
    sees (state planes L2-resident)."""
    T = obs_ring.shape[0]
    graph = env.capture_rollout(actions[:T].contiguous(), obs_ring, reward[:T], flags[:T])
    reps = max(1, steps // T)
    graph.replay()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    s.record()
    for _ in range(reps):
        graph.replay()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e), reps * T


def timing_floor(torch, env, flush, reps=200):
    """What an event pair reads around an (almost) empty kernel after the same flush: the fixed cost of one timed region."""
    out = []
    for _ in range(reps):
        flush()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        env.episode_stats_tensor()
        b.record()
        out.append((a, b))
    torch.cuda.synchronize()
    ts = sorted(a.elapsed_time(b) for a, b in out)
    return ts[len(ts) // 2]


def make_buffers(torch, env, n, device, seed, ring=FRAGMENT):
    g = torch.Generator(device=device).manual_seed(seed)
    lo, hi = (torch.as_tensor(x, device=device) for x in (env.action_space.low, env.action_space.high))
    n_act = ring
    actions = lo + torch.rand((n_act, n, DOF), device=device, generator=g) * (hi - lo)     # uniform in the action space
    # rollout-fragment style observation ring: consecutive steps write different slots; rows padded to a multiple of 4
    n_obs = max(2, min(ring, (1 << 30) // (n * OBS_DIM * 4)))
    n_pad = (n + 3) // 4 * 4
    obs_ring = torch.empty((n_obs, n_pad, OBS_DIM), dtype=torch.float32, device=device)[:, :n]
    reward = torch.empty((n_act, n), dtype=torch.float32, device=device)
    flags = torch.empty((n_act, n), dtype=torch.uint8, device=device)
    return actions, obs_ring, reward, flags


DUMP_BYTES_MAX = 64 << 20


def dump_outputs(out_dir, arrays, seed=0):
    """Write each array of `arrays` (name -> [N, ...], one row per env) as out_dir/<name>.npy: float64 stays float64, every
    other dtype becomes float32.  When the rows do not fit in DUMP_BYTES_MAX, the same fixed, seeded sample of rows is
    taken from every array and the sampled env indices are written as env_index.npy (float64)."""
    import numpy as np
    arrays = {k: np.asarray(v) for k, v in arrays.items()}
    arrays = {k: v if v.dtype == np.float64 else v.astype(np.float32) for k, v in arrays.items()}
    n = len(next(iter(arrays.values())))
    row_bytes = sum(v[:1].nbytes for v in arrays.values())
    if n * row_bytes > DUMP_BYTES_MAX:
        keep = (DUMP_BYTES_MAX - 4096 * (len(arrays) + 1)) // (row_bytes + 8)       # 4 KiB for each .npy header
        rows = np.sort(np.random.default_rng(seed).choice(n, keep, replace=False))
        arrays = {k: v[rows] for k, v in arrays.items()}
        arrays["env_index"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, v in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(v))


def pre_age(torch, env, limit, seed):
    """Give every env a random age in [0, limit): the timed region then runs the steady-state mix of a long rollout, with
    n / limit TimeLimit truncations + in-kernel Philox auto-resets per step, instead of `limit` reset-free steps."""
    g = torch.Generator(device=env.device).manual_seed(seed)
    env.set_state(t=torch.randint(0, limit, (env.n_envs,), device=env.device, generator=g, dtype=torch.int32))


def ours_arm(args):
    import torch
    import torch.distributed as dist
    from pioneer_b200 import BatchConfig, BatchedPioneerEnv, SimulationConfig, demo_obstacles
    from pioneer_b200.distributed import reduce_episode_stats, summarize

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback "
                         "(use --impl reference for the CPU arm)")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries exactly ONE JSON line: native libraries (NCCL prints its version banner and NCCL_DEBUG lines on fd 1)
    # go to stderr
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    if world == 1 and args.gpus > 1:
        raise SystemExit("bench.py: for --gpus N > 1 launch with torch.distributed.run, one rank per GPU")
    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)
    from pioneer_b200.distributed import bind_to_gpu_numa_node
    numa_node = bind_to_gpu_numa_node(local_rank) if world > 1 else None    # pinned e2e buffers on the GPU's socket
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)

    n = args.envs_per_gpu
    LIMIT = 500
    env = BatchedPioneerEnv(n, device=device, seed=0, env_id_base=rank * n,
                            batch_config=BatchConfig(max_episode_steps=LIMIT, auto_reset=True, obs_mode="terminal"))
    pre_age(torch, env, LIMIT, seed=100 + rank)
    actions, obs_ring, reward, flags = make_buffers(torch, env, n, device, seed=rank)
    flush_buf = torch.empty(L2_FLUSH_BYTES // 4, dtype=torch.float32, device=device)
    if args.flush == "write":
        def flush():
            flush_buf.zero_()
    elif args.flush == "none":
        def flush():
            pass
    else:
        flush_src = torch.zeros(L2_FLUSH_BYTES // 4, dtype=torch.float32, device=device)

        def flush():
            flush_buf.zero_()
            flush_src.sum()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for _ in range(3):                                       # communicator set-up and warm-up outside every timed region
        reduce_episode_stats(env.episode_stats_tensor())
    sampler = ClockSampler(local_rank) if rank == 0 else None
    # ---- device-resident throughput: `value` ---------------------------------------------------------
    env.episode_stats(clear=True)
    barrier()
    if sampler:
        sampler.start()
    wall0 = time.perf_counter()
    kernel_ms, per_frag = time_fragments(torch, env, actions, obs_ring, reward, flags, args.steps, args.warmup, flush)
    launches = time_fragments.launches
    barrier()
    wall_s = time.perf_counter() - wall0
    kernel_ms_max = max_over_ranks(kernel_ms)
    total_envs = n * world
    value = total_envs * args.steps / (kernel_ms_max / 1e3)
    clocks = sampler.finish() if sampler else None
    if args.dump_outputs and rank == 0:                      # the last timed step's slot, before later timings reuse it
        last = per_frag[-1][1] - 1
        dump_outputs(args.dump_outputs, {"obs": obs_ring[last].cpu(), "reward": reward[last].cpu(),
                                         "flags": flags[last].cpu()})
    # the path's one exchange: episode statistics, once per iteration (distributed.IterationSync).  Within a node it is ONE
    # kernel per rank over NVLink peer memory (pnr_iteration_sync: snapshot + stores into every rank's window + flags + merge),
    # replayed from a CUDA graph; the NCCL form (snapshot kernel + all_gather_into_tensor + merge kernel, eager) is timed
    # beside it.  Median of 20 back-to-back exchanges after warm-up, max over ranks.
    from pioneer_b200.distributed import IterationSync
    stats = reduce_episode_stats(env.episode_stats_tensor()).clone()       # the window of the timed region, for the line

    def time_sync(sync):
        for _ in range(3):
            sync()
        barrier()
        evs = []
        for _ in range(20):
            a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a_.record()
            sync()
            b_.record()
            evs.append((a_, b_))
        torch.cuda.synchronize()
        return max_over_ranks(sorted(a_.elapsed_time(b_) for a_, b_ in evs)[10])

    it_sync = IterationSync(env, None, None, clear=False, cuda_graph=True)
    stats_ms = time_sync(it_sync)
    exchange = {"transport": it_sync.transport, "cuda_graph": it_sync._graph is not None, "ms": stats_ms,
                "timed_out": it_sync.timed_out()}
    nccl_sync = IterationSync(env, None, None, clear=False, cuda_graph=False, transport="nccl")
    exchange["nccl_eager_ms"] = time_sync(nccl_sync)
    # both merge in rank order: bit-identical; NCCL's all-reduce may associate the float64 sums differently
    assert torch.equal(it_sync.merged[:8], nccl_sync.merged[:8]), "the peer-memory exchange disagrees with all-gather + merge"
    assert torch.allclose(it_sync.merged[:8], stats, rtol=1e-12, atol=0.0), "the exchange disagrees with the all-reduce"
    del nccl_sync

    # ---- the round-1 method on the same env: one event pair and one flush per STEP ----------------------
    k1 = min(args.steps, 1000)
    step_ms, per_step = time_device_steps(torch, env, actions, obs_ring, reward, flags, k1, min(args.warmup, 20), flush)
    step_ms = max_over_ranks(step_ms)
    srt = sorted(per_step)
    # ---- no flush at all, replayed from a CUDA graph (what a device-resident rollout loop sees) ------------
    barrier()
    graph_ms, graph_steps = time_graph(torch, env, actions, obs_ring, reward, flags, args.steps)
    graph_ms = max_over_ranks(graph_ms)
    floor_ms = timing_floor(torch, env, flush)

    # ---- end to end through the public host API: pinned host actions in, obs/reward/done out ------------
    # (a) the asynchronous double-buffered call with the compact row layout: D2H of step k overlaps H2D + kernel of step
    #     k + 1; the caller's next action does not wait for the observation still in flight (random actions here)
    # (b) the synchronous full-row call of round 1 (pnr_step_host)
    e2e_steps = min(args.steps, 300)
    host_actions = [torch.empty((n, DOF), dtype=torch.float32, pin_memory=True).copy_(actions[i % actions.shape[0]])
                    for i in range(4)]
    for k in range(3):
        env.step_host(host_actions[k % 4])
    barrier()
    t0 = time.perf_counter()
    checksum = 0.0
    for k in range(e2e_steps):
        _, h_reward, _ = env.step_host(host_actions[k % 4])
        checksum += float(h_reward[0])
    torch.cuda.synchronize()
    e2e_sync_s = max_over_ranks(time.perf_counter() - t0)
    env.step_host_begin(host_actions[0], compact=True)          # warm-up: both staging slots, both pinned buffer sets
    for k in range(6):
        env.step_host_begin(host_actions[(k + 1) % 4], compact=True)
        env.step_host_end()
    env.step_host_end()
    barrier()
    t0 = time.perf_counter()
    env.step_host_begin(host_actions[0], compact=True)
    for k in range(e2e_steps):
        if k + 1 < e2e_steps:
            env.step_host_begin(host_actions[(k + 1) % 4], compact=True)
        _, h_reward, _ = env.step_host_end()
        checksum += float(h_reward[0])                       # the result is read on the host every step
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    e2e_value = total_envs * e2e_steps / e2e_s

    peak, peak_src = measured_hbm_peak()
    avg_ms = kernel_ms / args.steps                      # this rank's kernel, per launch
    achieved = BYTES_PER_ENV_STEP * n / (avg_ms / 1e3) / 1e9
    traffic, traffic_steps, traffic_src, src_hash = ncu_traffic(env._lib, n)
    frag_ms = sorted(ms / t for ms, t in per_frag)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": kernel_ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"BASELINE.json configs[2]: batched reach env, {n} envs per GPU, joint limits, "
                               "TimeLimit 500, in-kernel auto-reset, uniform random actions in [-a_max, a_max]",
                   "envs_per_gpu": n, "total_envs": total_envs, "mode": "kinematic (the reference env)",
                   "arith": "f32", "obs": f"float32[N,137] terminal observations, {obs_ring.shape[0]}-slot rollout ring",
                   "env_ages": f"uniform in [0, {LIMIT}): ~n/{LIMIT} TimeLimit truncations + Philox auto-resets per step",
                   "l2": ("NOT FLUSHED (profiling run, not a bench value); " if args.flush == "none" else
                          f"flushed between timed fragments ({L2_FLUSH_BYTES >> 20} MiB memset"
                          + (" then a 512 MiB read sweep" if args.flush != "write" else "") + ", untimed); ")
                         + f"a fragment = {FRAGMENT} consecutive steps in ONE kernel launch (pnr_step_many: every CTA runs the "
                           "steps on its own tiles), each fragment timed by its own CUDA-event pair on the launching stream; within a "
                           f"fragment the {n * 96 // 1000000} MB of env state stay L2-resident as in any rollout loop, the "
                           f"{obs_ring.shape[0]} x {n * OBS_DIM * 4 // 1000000} MB observation slots do not fit",
                   "parallelism": f"env-sharded x{world}, no data-path collective; one statistics exchange per iteration "
                                  "(stats_exchange: a peer-memory kernel within the node, NCCL all-gather + merge otherwise)"},
        "substeps_per_sec": value * FRAME_SKIP,
        "fragment_steps": FRAGMENT,
        "fragment_ms_per_step_percentiles": {"p5": frag_ms[len(frag_ms) // 20], "p50": frag_ms[len(frag_ms) // 2],
                                             "p95": frag_ms[(len(frag_ms) * 19) // 20]},
        "timing_floor_ms": floor_ms,
        "per_step_flushed": {"note": "round-1 method: one event pair and one L2 flush per step", "steps": k1,
                             "ms_per_step": step_ms / k1, "value": total_envs * k1 / (step_ms / 1e3),
                             "frac": (BYTES_PER_ENV_STEP * n / (step_ms / k1 / 1e3) / 1e9) / peak,
                             "p5": srt[len(srt) // 20], "p50": srt[len(srt) // 2], "p95": srt[(len(srt) * 19) // 20]},
        "value_l2_warm_cuda_graph": total_envs * graph_steps / (graph_ms / 1e3),
        "ms_per_step_l2_warm_cuda_graph": graph_ms / graph_steps,
        "stats_allreduce_ms": stats_ms,
        "stats_exchange": exchange,
        "episode_stats": summarize(stats),
        "wall_s_timed_region_incl_flush": wall_s,
        "gpu_launches": launches,
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": n * DOF * 4,
                "d2h_bytes_per_step": n * (101 * 4 + 4 + 1), "steps": e2e_steps,
                "api": "BatchedPioneerEnv.step_host_begin / step_host_end -> pnr_step_host_begin(PNR_HOST_COMPACT) / _end: pinned "
                       "host buffers, copies inside the timed region, two steps in flight (the D2H of step k overlaps H2D + "
                       "kernel of step k + 1), 101-column rows (the 36 constant columns are delivered once)",
                "sync_full_rows": {"value": total_envs * e2e_steps / e2e_sync_s, "d2h_bytes_per_step": n * (OBS_DIM * 4 + 4 + 1),
                                   "api": "BatchedPioneerEnv.step_host -> pnr_step_host (synchronous, 137-column rows)"},
                # what the host links of the whole box carried: if this stops growing with N the box, not the path, is the limit
                "host_link_gb_per_s_all_ranks": e2e_value * (DOF * 4 + 101 * 4 + 4 + 1) / 1e9,
                "numa_node_rank0": numa_node,
                "timer": "host perf_counter around the calls, max over ranks"},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_capture": traffic_src, "source_hash": src_hash,
                     "kernel": "pnr_step_kernel<F32,TERMINAL>",
                     # one launch = one rollout fragment: `achieved` = algorithmic bytes of a launch / its duration, which is
                     # bytes_per_env_step * envs / ms_per_step; `traffic` is ncu's DRAM bytes of one such launch
                     "bytes_per_env_step": BYTES_PER_ENV_STEP, "units_per_launch": n * min(FRAGMENT, args.steps),
                     "steps_per_launch": min(FRAGMENT, args.steps), "traffic_steps_per_launch": traffic_steps,
                     "algorithmic_bytes_per_launch": BYTES_PER_ENV_STEP * n * min(FRAGMENT, args.steps),
                     "peak_source": peak_src},
    }
    del it_sync                                              # its graph points into the handle
    env.close()
    del obs_ring, actions

    k_extra = min(args.steps, 200)

    def timed_extra(make_env, seed, steps=None, fragment=FRAGMENT):
        e = make_env()
        pre_age(torch, e, LIMIT, seed)
        a, o, r, f = make_buffers(torch, e, e.n_envs, device, seed=seed)
        ks = steps or k_extra
        barrier()
        ms, _ = time_fragments(torch, e, a, o, r, f, ks, min(args.warmup, 16), flush, fragment)
        ms = max_over_ranks(ms)
        e.close()
        del a, o, r, f
        return ms / ks

    # ---- Tier-B dynamic mode (ABA + PD control, 10 substeps per env step) at every N ---------------------------
    def dyn_env(m, obstacles=(), penalty=0.0):
        return lambda: BatchedPioneerEnv(m, device=device, seed=0, env_id_base=rank * m,
                                         simulation_config=SimulationConfig(gravity=9.81),
                                         batch_config=BatchConfig(mode="dynamic", kp=2000.0, kd=500.0, torque_scale=1e5,
                                                                  max_episode_steps=LIMIT, obstacles=list(obstacles),
                                                                  contact_penalty=penalty))

    def dyn_record(m, ms, kernel):
        v = world * m / (ms / 1e3)
        tf = (v / world) * DYN_FLOP_PER_ENV_STEP / 1e12
        return {"workload": f"{m} envs per GPU, gravity 9.81, PD position control (kp 2000, kd 500), set points uniform in the "
                            f"joint range, {FRAME_SKIP} ABA substeps per env step, TimeLimit 500 + auto-reset",
                "ms_per_step": ms, "value": v, "unit": UNIT, "substeps_per_sec": FRAME_SKIP * v,
                "parity": "float64 oracle at this size (tests/test_gpu_dynamic_parity.py), unpinned vs PyBullet",
                "roofline": {"bound": "fp32", "achieved": tf, "peak": FP32_PEAK_TFLOPS, "unit": "TFLOP/s",
                             "frac": tf / FP32_PEAK_TFLOPS, "flop_per_env_step": DYN_FLOP_PER_ENV_STEP,
                             "fp32_issue_frac": (v / world) * DYN_FP_INSTR_PER_ENV_STEP / (FP32_PEAK_TFLOPS / 2 * 1e12),
                             "peak_source": "tools/fma_peak.py on this pool's B200 (FMA = 2 flop)", "kernel": kernel,
                             # context: the same kernel against what its own FP32 instruction stream can issue at best,
                             # given the measured three-register FFMA rate (profiles/r02_fp32_forms.md)
                             "operand_bound": {
                                 "env_steps_per_s": SM_SUBPARTITIONS * SM_CLOCK_HZ / DYN_OPERAND_BOUND_CLOCKS * 32,
                                 "frac": (v / world) / (SM_SUBPARTITIONS * SM_CLOCK_HZ / DYN_OPERAND_BOUND_CLOCKS * 32),
                                 "three_register_ffma_per_clock_per_smsp": 0.711}}}

    if not args.no_extras:
        line["dynamic_mode"] = dyn_record(n, timed_extra(dyn_env(n), 2), "pnr_step_dynamic_kernel<TERMINAL,false,PIONEER_ISO>")
        # ---- BASELINE configs[3]: reach with obstacles, 16,384 envs per GPU --------------------------------------
        m = 16384
        obst = demo_obstacles()
        ms_k = timed_extra(lambda: BatchedPioneerEnv(m, device=device, seed=0, env_id_base=rank * m,
                                                     batch_config=BatchConfig(max_episode_steps=LIMIT, obstacles=obst,
                                                                              contact_penalty=0.5, random_box=True)), 4)
        ms_d = timed_extra(dyn_env(m, obst, 0.5), 5)
        line["obstacles"] = {
            "workload": f"BASELINE.json configs[3]: {m} envs per GPU, 5 link capsules vs ground plane / box / sphere (exact "
                        "segment distances), contact penalty in the reward; kinematic: box redrawn per episode (random_box)",
            "kinematic": {"ms_per_step": ms_k, "value": world * m / (ms_k / 1e3), "unit": UNIT},
            "dynamic": {"ms_per_step": ms_d, "value": world * m / (ms_d / 1e3), "unit": UNIT},
            "parity": "oracle/reach_oracle.c and oracle/dynamics_oracle.c at this size (tests/test_gpu_obstacles.py, "
                      "tests/test_gpu_dynamic_parity.py), geometry invented: unpinned"}
        # ---- BASELINE configs[4]: the rollout loop (filter + policy stub + env step) at 131,072 envs per GPU ----------
        line["rollout"] = rollout_loop(torch, dist, device, rank, world, max_over_ranks, barrier)

    # ---- env-count sweep (N=1 only): the metric is quoted at 4K..1M envs --------------------------------
    if world == 1 and not args.no_sweep:
        sweep = []
        for m in (4096, 16384, 131072, 1048576):
            e = BatchedPioneerEnv(m, device=device, seed=0, batch_config=BatchConfig(max_episode_steps=LIMIT))
            pre_age(torch, e, LIMIT, 7)
            a, o, r, f = make_buffers(torch, e, m, device, seed=1)
            k_steps = min(args.steps, 1000)
            ms, _ = time_fragments(torch, e, a, o, r, f, k_steps, min(args.warmup, 24), flush)
            ms_1, _ = time_device_steps(torch, e, a, o, r, f, min(k_steps, 300), 10, flush)
            gbs = BYTES_PER_ENV_STEP * m / (ms / k_steps / 1e3) / 1e9
            sweep.append({"envs": m, "ms_per_step": ms / k_steps, "value": m * k_steps / (ms / 1e3),
                          "ms_per_step_flushed_every_step": ms_1 / min(k_steps, 300), "achieved_gbs": gbs, "frac": gbs / peak})
            e.close()
            del a, o, r, f
        line["sweep"] = sweep
        big = sweep[-1]
        tr, tr_steps, tr_src, _ = ncu_traffic(env._lib, big["envs"])
        line["roofline_large_batch"] = {
            "bound": "hbm", "achieved": big["achieved_gbs"], "peak": peak, "unit": "GB/s", "frac": big["frac"],
            "traffic": tr, "traffic_capture": tr_src, "traffic_steps_per_launch": tr_steps,
            "kernel": "pnr_step_kernel<F32,TERMINAL>", "bytes_per_env_step": BYTES_PER_ENV_STEP,
            "units_per_launch": big["envs"] * 2, "steps_per_launch": 2, "peak_source": peak_src}
        ms_big = timed_extra(dyn_env(1048576), 6, steps=min(args.steps, 64))
        line["dynamic_mode_large_batch"] = dyn_record(1048576, ms_big, "pnr_step_dynamic_kernel<TERMINAL,false,PIONEER_ISO>")

    # ---- N2: fused observation normaliser (one pass: push statistics + normalise in place) -------------------------
    if world == 1 and not args.no_sweep:
        from pioneer_b200.obs_filter import MeanStdObsFilter
        filt = []
        for m in (args.envs_per_gpu, 1048576):
            e = BatchedPioneerEnv(m, device=device, seed=0)
            flt_ = MeanStdObsFilter(e)
            ring = torch.randn((max(2, min(8, (1 << 30) // (m * OBS_DIM * 4))), m, OBS_DIM), device=device)
            for k in range(3):
                flt_(ring[k % ring.shape[0]])
            flt_.sync()
            evs = []
            for k in range(50):
                flush()
                a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a_.record(); flt_(ring[k % ring.shape[0]]); b_.record()
                evs.append((a_, b_))
            torch.cuda.synchronize()
            ms = sum(a_.elapsed_time(b_) for a_, b_ in evs) / len(evs)
            gbs = 2 * OBS_DIM * 4 * m / (ms / 1e3) / 1e9
            # the same normalisation fused into the step kernel (pnr_filter_fuse): no second pass over the observations
            flt_.set_fused(True)
            a2, o2, r2, f2 = make_buffers(torch, e, m, device, seed=3)
            k2 = min(args.steps, 304)
            ms_fused, _ = time_fragments(torch, e, a2, o2, r2, f2, k2, 16, flush)
            flt_.set_fused(False)
            ms_plain, _ = time_fragments(torch, e, a2, o2, r2, f2, k2, 16, flush)
            filt.append({"rows": m, "ms": ms, "rows_per_sec": m / (ms / 1e3), "achieved_gbs": gbs, "frac": gbs / peak,
                         "bytes_per_row": 2 * OBS_DIM * 4, "step_ms_plain": ms_plain / k2,
                         "step_ms_fused_normaliser": ms_fused / k2, "step_plus_filter_pass_ms": ms_plain / k2 + ms})
            e.close()
            del ring, a2, o2, r2, f2
        line["obs_filter"] = filt

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            line["cpu_baseline"] = cpu_baseline_subprocess()
        except Exception as exc:  # noqa: BLE001
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": _host_cores(), "kind": "port",
                                    "sample": f"failed: {exc!r}"}
    if rank == 0:
        os.write(json_fd, (json.dumps(_finite(line)) + "\n").encode())
    if world > 1:
        # teardown must never outlive the measurement: graphs and envs go first, and a communicator that does not shut down
        # within 30 s (seen once with NCCL kernels still referenced by live CUDA graphs) is abandoned, not waited for
        import gc
        import threading
        gc.collect()
        torch.cuda.synchronize()
        dist.barrier()
        guard = threading.Timer(30.0, lambda: os._exit(0))
        guard.daemon = True
        guard.start()
        dist.destroy_process_group()
        guard.cancel()


def rollout_loop(torch, dist, device, rank, world, max_over_ranks, barrier, n=131072, fragment=8, iters=12):
    """BASELINE.json configs[4]: observation filter (fused into the step) -> 137-256-256-12 policy stub (torch / cuBLAS:
    RLlib's side of the boundary) -> sampled action -> fused env step, fragments replayed from a CUDA graph, ONE collective
    per iteration (episode statistics + filter delta packed into one all-gather, merged by one kernel).  1,048,576 envs on
    8 GPUs.  Device time from CUDA events, max over ranks."""
    from pioneer_b200 import BatchConfig, BatchedPioneerEnv
    from pioneer_b200.distributed import summarize
    from pioneer_b200.rollout import RolloutWorker
    env = BatchedPioneerEnv(n, device=device, seed=0, env_id_base=rank * n, batch_config=BatchConfig(max_episode_steps=500))
    torch.cuda.manual_seed(1234 + rank)
    worker = RolloutWorker(env, fragment_length=fragment, seed=rank, cuda_graph=True)
    worker.collect()                               # the first fragment starts with env.reset()
    pre_age(torch, env, 500, 11 + rank)            # ... then the envs get their steady-state ages
    for _ in range(3):
        worker.collect()
        worker.sync(summary=False)
    barrier()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(iters):
        worker.collect()
        stats = worker.sync(summary=False)         # stays on the device: the loop never waits for the GPU
    e.record()
    torch.cuda.synchronize()
    ms = max_over_ranks(s.elapsed_time(e))
    steps = iters * fragment
    out = {"workload": f"BASELINE.json configs[4]: {n} envs per GPU ({world * n} in total), fragment length {fragment}, fused "
                       "observation filter, bf16 137-256-256-12 policy stub, CUDA-graph fragments, one packed exchange (statistics + filter delta) per "
                       "iteration; the policy sees the reset observation after every done (pnr_observe_done)",
           "value": world * n * steps / (ms / 1e3), "unit": UNIT, "ms_per_env_step_batch": ms / steps, "iterations": iters,
           "episode_stats": summarize(stats)}
    env.close()
    return out


def _finite(x):
    """Strict JSON: NaN / inf become null."""
    if isinstance(x, float):
        return x if math.isfinite(x) else None
    if isinstance(x, dict):
        return {k: _finite(v) for k, v in x.items()}
    if isinstance(x, (list, tuple)):
        return [_finite(v) for v in x]
    return x


def main():
    args = parse_args()
    if args.impl == "reference":
        reference_arm(args)
    else:
        ours_arm(args)


if __name__ == "__main__":
    main()
