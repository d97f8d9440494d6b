"""Host-side launch layer: sequence sharding, and the N>1 path with a world_size-2 gloo run on CPU."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from comet_pose_estimation_b200 import launch


def test_shard_indices_partition():
    for n in (0, 1, 7, 16, 33):
        for world in (1, 2, 3, 8):
            seen = []
            for r in range(world):
                idx = launch.shard_indices(n, r, world)
                assert idx == sorted(idx) and all(i % world == r for i in idx)
                seen += idx
            assert sorted(seen) == list(range(n))
            sizes = [len(launch.shard_indices(n, r, world)) for r in range(world)]
            assert max(sizes) - min(sizes) <= 1


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, n_items, out_dir):
    os.environ.update(RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE=str(world), MASTER_ADDR="127.0.0.1",
                      MASTER_PORT=str(port))
    env = launch.init_distributed(backend="gloo")
    assert env["RANK"] == rank and dist.get_world_size() == world
    rng = np.random.default_rng(0)
    items = [rng.standard_normal((4, 3)).astype(np.float32) for _ in range(n_items)]
    local = launch.run_sharded(items, lambda a: float(a.sum()))       # data path: no communication
    assert sorted(local) == launch.shard_indices(n_items, rank, world)
    allr = launch.gather_results(local, n_items)                      # the one collective, at the end
    thr = launch.throughput_sequences_per_s(len(local), 2.0 + rank)   # slowest rank sets the time
    if rank == 0:
        want = [float(a.sum()) for a in items]
        assert allr == want
        assert abs(thr - n_items / (2.0 + world - 1)) < 1e-9
        open(os.path.join(out_dir, "ok"), "w").write("1")
    else:
        assert allr is None
    dist.destroy_process_group()


def test_two_rank_gloo_shard_and_gather(tmp_path, monkeypatch):
    world, n_items = 2, 7
    # a CPU run whatever the machine has: with GPUs visible, init_distributed binds rank r to cuda:r, which a machine
    # with fewer GPUs than ranks does not have
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "")
    mp.spawn(_worker, args=(world, _free_port(), n_items, str(tmp_path)), nprocs=world, join=True)
    assert (tmp_path / "ok").exists()


def test_single_process_paths():
    local = launch.run_sharded(list(range(5)), lambda x: x * x, rank=0, world=1)
    assert launch.gather_results(local, 5) == [0, 1, 4, 9, 16]
    assert launch.throughput_sequences_per_s(10, 2.0) == 5.0


@pytest.mark.gpu
def test_cuda_graph_replay_matches_eager():
    import comet_pose_estimation_b200 as cb

    torch.manual_seed(0)
    fm = torch.randn(1, 4, 128, 64, 64, device="cuda")
    blk = cb.CorrBlock(fm, num_levels=5, radius=4)
    tdim = cb.transformer_dim(5, 4, 128, False)
    c0 = torch.rand(1, 4, 100, 2, device="cuda") * 63
    f0 = torch.randn(1, 4, 100, 128, device="cuda")
    tok = cb.TrackTokenizer(blk, c0[:, 0], tdim)
    out = torch.empty(1, 100, 4, tdim, device="cuda")
    runner = launch.CudaGraphRunner(lambda c, f: tok.tokens(c, f, out=out), c0.clone(), f0.clone())
    for seed in (1, 2):
        g = torch.Generator(device="cuda").manual_seed(seed)
        c = c0 + torch.randn(c0.shape, device="cuda", generator=g)
        c[:, 0] = c0[:, 0]
        f = torch.randn(f0.shape, device="cuda", generator=g)
        got = runner(c, f).clone()
        want = tok.tokens(c, f)
        assert torch.equal(got, want)


def test_numa_binding_is_a_noop_without_a_gpu_or_sysfs():
    """bind_to_gpu_numa_node never raises: without a CUDA device / sysfs entry it changes nothing and returns None."""
    import os

    from comet_pose_estimation_b200 import launch

    before = sorted(os.sched_getaffinity(0))
    prev = launch.bind_to_gpu_numa_node(0)
    if prev is not None:  # a GPU box with several NUMA nodes: restore
        os.sched_setaffinity(0, prev)
    assert sorted(os.sched_getaffinity(0)) == before
