"""Multi-GPU sharding of the env batch and the one collective the path has.

Envs are independent: a job of ``total_envs`` is cut into contiguous ranges of global env ids, one
per rank / GPU, with no data-path communication.  Once per training iteration the per-GPU episode
statistics (the columns the reference CLI prints, cli.py:32-38) are reduced with NCCL over
NVLink: SUM over the counters and MAX over (max_return, -min_return).  The reference moves the same
numbers from its Ray rollout workers to the trainer (pioneer/launch/pioneer_knm_train.py:49).
"""
from __future__ import annotations

from typing import Dict, Optional, Tuple

import torch
import torch.distributed as dist

from . import _cabi
from .batched_env import STATS_FIELDS


def bind_to_gpu_numa_node(device_index: int) -> Optional[int]:
    """Pin this process to the CPUs of the NUMA node the GPU hangs off, BEFORE any pinned host buffer is allocated, so
    that the host side of the H2D / D2H copies (pnr_step_host) is local memory.  One rank per GPU on a two-socket box
    otherwise lands its pinned buffers wherever the scheduler started it.  Returns the node, or None if unknown."""
    import os
    try:
        bus = torch.cuda.get_device_properties(device_index).pci_bus_id
        dom = getattr(torch.cuda.get_device_properties(device_index), "pci_domain_id", 0)
        dev = torch.cuda.get_device_properties(device_index).pci_device_id
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{dev:02x}.0/numa_node"
        node = int(open(path).read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = cpus & set(os.sched_getaffinity(0))
        if not allowed:
            return None
        os.sched_setaffinity(0, allowed)
        return node
    except Exception:  # noqa: BLE001 - sysfs layout / permissions differ between boxes: binding is best effort
        return None


def shard_range(total_envs: int, rank: int, world_size: int) -> Tuple[int, int]:
    """(env_id_base, n_local): contiguous split, the first ``total % world`` ranks get one more."""
    assert 0 <= rank < world_size and total_envs >= world_size
    q, r = divmod(total_envs, world_size)
    n_local = q + (1 if rank < r else 0)
    base = rank * q + min(rank, r)
    return base, n_local


def _gather_merge(packed: torch.Tensor, gathered: torch.Tensor, out: torch.Tensor,
                  group: Optional[dist.ProcessGroup] = None, stream: Optional[int] = None) -> torch.Tensor:
    """Every rank's ``packed`` vector all-gathered into ``gathered`` [world, len] (one NCCL all-gather on the GPU, gloo on
    the CPU; none at world 1, where ``gathered`` is ``packed`` itself) and merged into ``out`` [len]: SUM over the counters
    and extras, MAX / MIN over slots 4 / 5.  On a GPU the merge is ONE kernel of the library (pnr_stats_merge_device) on
    ``stream``, which belongs to the current device; on the CPU plain torch."""
    world, k = gathered.shape
    if world > 1:
        if packed.is_cuda:
            dist.all_gather_into_tensor(gathered, packed, group=group)
        else:
            dist.all_gather(list(gathered.unbind(0)), packed, group=group)
    if gathered.is_cuda:
        _cabi.check(_cabi.load().pnr_stats_merge_device(gathered.data_ptr(), world, k, out.data_ptr(), stream),
                    "pnr_stats_merge_device")
        return out
    torch.sum(gathered, 0, out=out)
    out[4] = gathered[:, 4].max()
    out[5] = gathered[:, 5].min()
    return out


def reduce_packed(stats_local: torch.Tensor, extra_local: Optional[torch.Tensor] = None,
                  group: Optional[dist.ProcessGroup] = None):
    """ONE collective for everything a rollout worker exchanges per iteration: the float64[8] episode statistics (SUM /
    MAX / MIN slots) and an optional additive float64 vector (the observation filter's delta) are packed, all-gathered
    into one [world, len] tensor, and reduced by one kernel.  Returns (stats, extra)."""
    assert stats_local.dtype == torch.float64 and stats_local.numel() == len(STATS_FIELDS)
    k = len(STATS_FIELDS)
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return stats_local.clone(), (None if extra_local is None else extra_local.clone())
    packed = (stats_local if extra_local is None else torch.cat([stats_local, extra_local])).contiguous()
    gathered = packed.new_empty((dist.get_world_size(group), packed.numel()))
    merged = torch.empty_like(packed)
    if packed.is_cuda:
        with torch.cuda.device(packed.device):
            _gather_merge(packed, gathered, merged, group, torch.cuda.current_stream().cuda_stream)
    else:
        _gather_merge(packed, gathered, merged, group)
    return merged[:k], (None if extra_local is None else merged[k:].contiguous())


def reduce_episode_stats(local: torch.Tensor, group: Optional[dist.ProcessGroup] = None) -> torch.Tensor:
    """The packed float64[8] statistics vector of all ranks: one all-gather + one merge kernel (any backend; NCCL on the
    GPUs).  Returns a new tensor on the same device."""
    return reduce_packed(local, None, group)[0]


class IterationSync:
    """Everything a rollout worker exchanges once per training iteration -- the episode statistics (optionally clearing the
    window) and, if given, the observation filter's delta -- with static buffers, over one of two transports:

    ``p2p``   pnr_iteration_sync: ONE kernel per rank does snapshot + exchange + merge (+ the filter's Chan merge) over
              NVLink peer memory: every rank stores its packed float64[8 (+ 275)] into every rank's window and releases a
              flag there, waits for its own flags, and merges in rank order, so all ranks end with bit-identical numbers.
              The windows are plain cudaMalloc memory opened across processes with CUDA IPC; torch.distributed only carries
              the 64-byte handles, once, at construction.  No NCCL call in the step, so with ``cuda_graph=True`` the launch
              is captured and replayed at any world size.
    ``nccl``  snapshot (pnr_stats_device [+ pnr_filter_delta_device]) -> all_gather_into_tensor (world > 1) ->
              pnr_stats_merge_device [+ pnr_filter_sync_device], the same gather-and-merge as ``reduce_packed``.  At
              world > 1 it always runs eagerly: a communicator whose kernels live graphs still reference does not shut down
              (DESIGN.md section 5).  At world 1 there is no collective and ``cuda_graph=True`` captures it.

    ``transport="auto"`` (default) uses p2p when every rank could open every other rank's window (same node, peer access)
    and nccl otherwise.  A capture that fails raises.  ``__call__`` returns the merged float64[8] statistics tensor
    (device, not synchronised; valid until the next call).  A p2p wait that exceeds ``timeout_s`` yields NaN statistics and
    ``timed_out()`` reports it (a kernel never spins for ever on a dead peer); the ranks' sequence numbers may then disagree,
    so the next object must be built with ``reconnect=True`` on every rank (it re-opens the windows and restarts the
    protocol; graphs captured by earlier objects on that env must not be replayed afterwards)."""

    def __init__(self, env, obs_filter=None, group: Optional[dist.ProcessGroup] = None, clear: bool = True,
                 cuda_graph: bool = False, transport: str = "auto", timeout_s: float = 20.0, reconnect: bool = False):
        self.env, self.filter, self.group, self.clear = env, obs_filter, group, bool(clear)
        self._cabi, self._lib = _cabi, env._lib
        k = len(STATS_FIELDS)
        self.k = k
        self.len = k + (_cabi.PNR_FILTER_DELTA_LEN if obs_filter is not None else 0)
        active = dist.is_available() and dist.is_initialized()
        self.world = dist.get_world_size(group) if active else 1
        self.rank = dist.get_rank(group) if active else 0
        self.timeout_ms = int(timeout_s * 1000)
        self._reconnect = bool(reconnect)
        dev = env.device
        self.packed = torch.zeros(self.len, dtype=torch.float64, device=dev)
        self.gathered = (torch.zeros((self.world, self.len), dtype=torch.float64, device=dev) if self.world > 1
                         else self.packed.view(1, -1))
        self.merged = torch.zeros(self.len, dtype=torch.float64, device=dev)
        self._graph = None
        if transport not in ("auto", "p2p", "nccl"):
            raise ValueError(f"unknown transport {transport!r}")
        self.transport = "p2p" if self.world == 1 and transport != "nccl" else transport
        if self.world > 1 and transport != "nccl":
            self.transport = "p2p" if self._connect_windows() else "nccl"
            if transport == "p2p" and self.transport != "p2p":
                raise RuntimeError("IterationSync(transport='p2p'): the ranks could not open each other's windows: "
                                   + self._connect_error)
        if cuda_graph and (self.transport == "p2p" or self.world == 1):
            with torch.cuda.device(dev):
                self._graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(self._graph):
                    self._run()

    def _connect_windows(self) -> bool:
        """Exchange the CUDA IPC handles of the windows (one all-gather of 64 bytes per rank) and open the peers' windows;
        True when EVERY rank succeeded (otherwise all of them fall back to the NCCL transport together)."""
        import ctypes as C
        c, lib, env = self._cabi, self._lib, self.env
        self._connect_error = ""
        # one connection per (handle, group): a second IterationSync on the same env reuses it -- re-opening the windows
        # would unmap the addresses an earlier object's captured graph still launches with.  Every rank takes this branch
        # together (the objects are constructed in the same order on all ranks, as any collective is).
        key = (self.world, self.rank, id(self.group) if self.group is not None else 0)
        if getattr(env, "_sync_connection", None) == key and not self._reconnect:
            return True
        ipc = (C.c_ubyte * c.PNR_SYNC_IPC_BYTES)()
        ok = 1
        if self.world > c.PNR_SYNC_MAX_PEERS or lib.pnr_sync_window_create(env._h, ipc) != 0:
            ok, self._connect_error = 0, (lib.pnr_last_error() or b"").decode() or "world > PNR_SYNC_MAX_PEERS"
        mine = torch.tensor(list(ipc), dtype=torch.uint8, device=env.device)
        everyone = torch.zeros(self.world * c.PNR_SYNC_IPC_BYTES, dtype=torch.uint8, device=env.device)
        dist.all_gather_into_tensor(everyone, mine, group=self.group)
        if ok:
            handles = (C.c_ubyte * (self.world * c.PNR_SYNC_IPC_BYTES))(*everyone.cpu().tolist())
            if lib.pnr_sync_window_connect(env._h, handles, self.world, self.rank) != 0:
                ok, self._connect_error = 0, (lib.pnr_last_error() or b"").decode()
        agreed = torch.tensor([ok], dtype=torch.int32, device=env.device)
        dist.all_reduce(agreed, op=dist.ReduceOp.MIN, group=self.group)      # doubles as the barrier: every window is open
        torch.cuda.synchronize(env.device)
        if int(agreed.item()) != 1 and not self._connect_error:
            self._connect_error = "another rank failed"
        if int(agreed.item()) == 1:
            env._sync_connection = key
        return int(agreed.item()) == 1

    def _run(self) -> None:
        env, c, lib = self.env, self._cabi, self._lib
        s = env._stream()
        if self.transport == "p2p":
            c.check(lib.pnr_iteration_sync(env._h, 1 if self.filter is not None else 0, 1 if self.clear else 0,
                                           self.merged.data_ptr(), self.timeout_ms, s), "pnr_iteration_sync")
            return
        c.check(lib.pnr_stats_device(env._h, self.packed.data_ptr(), 1 if self.clear else 0, s), "pnr_stats_device")
        if self.filter is not None:
            c.check(lib.pnr_filter_delta_device(env._h, self.packed.data_ptr() + 8 * self.k, s), "pnr_filter_delta_device")
        _gather_merge(self.packed, self.gathered, self.merged, self.group, s)
        if self.filter is not None:
            c.check(lib.pnr_filter_sync_device(env._h, self.merged.data_ptr() + 8 * self.k, s), "pnr_filter_sync_device")

    def __call__(self) -> torch.Tensor:
        with torch.cuda.device(self.env.device):
            if self._graph is not None:
                self._graph.replay()
            else:
                self._run()
        return self.merged[:self.k]

    def timed_out(self) -> bool:
        """True if a p2p exchange gave up waiting for a peer (synchronises the device)."""
        import ctypes as C
        flag = C.c_int(0)
        self._cabi.check(self._lib.pnr_sync_status(self.env._h, C.byref(flag)), "pnr_sync_status")
        return bool(flag.value)


def summarize(stats: torch.Tensor) -> Dict[str, float]:
    """episode_reward_max/min/mean, episode_len_mean, episodes_total (cli.py:32-38) from the packed vector."""
    s = [float(x) for x in stats.tolist()]
    n = s[0]
    if not n:      # no episode finished in the window: None (JSON null), never NaN / inf
        return {"episodes_total": 0.0, "episode_reward_mean": None, "episode_reward_std": None, "episode_reward_max": None,
                "episode_reward_min": None, "episode_len_mean": None, "env_steps": s[6], "reached_target": s[7]}
    mean = s[1] / n
    var = max(s[3] / n - mean * mean, 0.0)
    return {"episodes_total": n, "episode_reward_mean": mean, "episode_reward_std": var ** 0.5,
            "episode_reward_max": s[4], "episode_reward_min": s[5], "episode_len_mean": s[2] / n, "env_steps": s[6],
            "reached_target": s[7]}
