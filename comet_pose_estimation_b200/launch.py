"""Batch sharding / launch layer for the tracking hot path (replaces what HF ``accelerate`` does for the reference's
eval and train scripts: ``Accelerator(...)`` + ``accelerator.prepare(dataloader)``, comet/models/abl_ours.py:28,59,
train_e2epose2.py:47,83).

One process per GPU (``torchrun`` / ``torch.distributed``).  Inference is pure data parallelism over *sequences*:
rank r processes sequences r, r + W, r + 2W, ... with NO collective on the data path (tracks of one sequence are
never split across GPUs: the update transformer couples them through its virtual tracks).  Only the final metric /
result gather uses a collective.  Training adds exactly one NCCL all-reduce of the camera-predictor gradients per
step (DDP), which is outside this path.

Also here: ``CudaGraphRunner`` -- capture a fixed-shape piece of the loop (e.g. the fused token kernel, or a whole
refinement iteration) into a CUDA graph so that B=1 latency is not dominated by launch overhead.
"""
from __future__ import annotations

import os
from typing import Any, Callable, Dict, Iterable, List, Optional, Sequence

import torch
import torch.distributed as dist


def dist_env() -> Dict[str, int]:
    """RANK / LOCAL_RANK / WORLD_SIZE as set by torchrun (defaults: single process)."""
    return {k: int(os.environ.get(k, d)) for k, d in (("RANK", "0"), ("LOCAL_RANK", "0"), ("WORLD_SIZE", "1"))}


def init_distributed(backend: Optional[str] = None) -> Dict[str, int]:
    """Initialise torch.distributed from the torchrun environment (NCCL on GPU, gloo otherwise) and bind this
    process to its GPU.  Safe to call in a single-process run (no process group is created)."""
    env = dist_env()
    if torch.cuda.is_available():
        torch.cuda.set_device(env["LOCAL_RANK"])
    if env["WORLD_SIZE"] > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29511")
        backend = backend or ("nccl" if torch.cuda.is_available() else "gloo")
        kw = {}
        if backend == "nccl":
            kw["device_id"] = torch.device("cuda", env["LOCAL_RANK"])
        dist.init_process_group(backend, rank=env["RANK"], world_size=env["WORLD_SIZE"], **kw)
    return env


def bind_to_gpu_numa_node(local_rank: int) -> Optional[List[int]]:
    """Pin this process to the CPUs of the NUMA node its GPU hangs off (read from sysfs), so that pinned host buffers
    allocated afterwards are node-local and H2D copies of several ranks do not cross the socket interconnect.
    Returns the previous affinity (to restore with ``os.sched_setaffinity(0, prev)``) or None if nothing was changed
    (no sysfs entry, single node, not Linux)."""
    try:
        pr = torch.cuda.get_device_properties(local_rank)
        bus = f"{int(pr.pci_domain_id):04x}:{int(pr.pci_bus_id):02x}:{int(pr.pci_device_id):02x}.0"
    except Exception:
        try:
            import pynvml

            pynvml.nvmlInit()
            bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(local_rank)).busId
            bus = bus.decode() if isinstance(bus, bytes) else bus
        except Exception:
            return None
    try:
        bus = str(bus).lower()
        if len(bus.split(":")[0]) == 8:  # nvml reports a 32-bit domain
            bus = bus[4:]
        with open(f"/sys/bus/pci/devices/{bus}/numa_node") as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = []
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.extend(range(int(a), int(b or a) + 1))
        prev = sorted(os.sched_getaffinity(0))
        cpus = [c for c in cpus if c in prev]
        if not cpus or len(cpus) == len(prev):
            return None
        os.sched_setaffinity(0, cpus)
        return prev
    except Exception:
        return None


def shard_indices(n_items: int, rank: int, world: int) -> List[int]:
    """Sequences owned by ``rank``: r, r+W, r+2W, ... (round-robin keeps ranks within one item of each other)."""
    assert 0 <= rank < world
    return list(range(rank, n_items, world))


def run_sharded(items: Sequence[Any], fn: Callable[[Any], Any], rank: Optional[int] = None,
                world: Optional[int] = None) -> Dict[int, Any]:
    """Apply ``fn`` to this rank's shard of ``items``; returns {global index: result}.  No communication."""
    env = dist_env()
    rank = env["RANK"] if rank is None else rank
    world = env["WORLD_SIZE"] if world is None else world
    return {i: fn(items[i]) for i in shard_indices(len(items), rank, world)}


def run_sharded_batched(items: Sequence[Any], fn: Callable[[List[Any]], Sequence[Any]], batch_size: int,
                        rank: Optional[int] = None, world: Optional[int] = None) -> Dict[int, Any]:
    """``run_sharded`` for a batched ``fn``: this rank's round-robin shard is cut, in order, into batches of at most
    ``batch_size`` items; ``fn(list of items)`` returns one result per item.  Returns {global index: result}, the same
    mapping ``run_sharded`` returns, so ``gather_results`` applies unchanged."""
    assert batch_size >= 1
    env = dist_env()
    rank = env["RANK"] if rank is None else rank
    world = env["WORLD_SIZE"] if world is None else world
    mine = shard_indices(len(items), rank, world)
    out: Dict[int, Any] = {}
    for k in range(0, len(mine), batch_size):
        idx = mine[k:k + batch_size]
        res = list(fn([items[i] for i in idx]))
        assert len(res) == len(idx), f"batched fn returned {len(res)} results for {len(idx)} items"
        out.update(zip(idx, res))
    return out


def gather_results(local: Dict[int, Any], n_items: int) -> Optional[List[Any]]:
    """End-of-run gather of per-sequence results (small objects: metrics, poses) to rank 0, in global order.
    This is the only collective of the inference path."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return [local[i] for i in range(n_items)]
    parts: List[Optional[Dict[int, Any]]] = [None] * dist.get_world_size() if dist.get_rank() == 0 else None
    dist.gather_object(local, parts, dst=0)
    if dist.get_rank() != 0:
        return None
    merged: Dict[int, Any] = {}
    for p in parts:
        overlap = merged.keys() & p.keys()
        assert not overlap, f"sequences {sorted(overlap)} were processed by two ranks"
        merged.update(p)
    assert len(merged) == n_items, "some sequences were not processed"
    return [merged[i] for i in range(n_items)]


def throughput_sequences_per_s(n_local: int, elapsed_s: float) -> float:
    """Whole-job sequences/s: all ranks' sequences over the slowest rank's time (max over ranks)."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return n_local / elapsed_s
    dev = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend() == "nccl" else torch.device("cpu")
    t = torch.tensor([elapsed_s], dtype=torch.float64, device=dev)
    n = torch.tensor([float(n_local)], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dist.all_reduce(n, op=dist.ReduceOp.SUM)
    return float(n.item() / t.item())


class CudaGraphRunner:
    """Capture ``fn(*static_inputs)`` once, replay it with new data copied into the static buffers.

    ``fn`` must be shape-static and allocation-stable (e.g. ``tokenizer.tokens(coords, feats, out=out)``).  Three
    eager warm-up calls run first on a side stream (library handles, the kernel's shared-memory attribute and its
    status word are created outside the capture)."""

    def __init__(self, fn: Callable[..., Any], *static_inputs: torch.Tensor):
        self.inputs = static_inputs
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(3):
                fn(*static_inputs)
        torch.cuda.current_stream().wait_stream(side)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.output = fn(*static_inputs)

    def __call__(self, *new_inputs: torch.Tensor):
        for dst, src in zip(self.inputs, new_inputs):
            if src is not dst:
                dst.copy_(src, non_blocking=True)
        self.graph.replay()
        return self.output
