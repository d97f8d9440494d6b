"""Sequences per second of ``TrackerPredictor.track_batch`` (ragged batches) against a loop of ``track()`` over the same
sequences, on one GPU.

    python scripts/ragged_batch_time.py [--seqs 16] [--reps 2] [--out result.json]

Workload: 16-frame 512x512 sequences, seeded random images, N_b drawn from a seeded U[256, 512] (what COMET's eval loop
keeps per sequence); default configuration weights (timing does not depend on their values).  For batch sizes 1 / 2 / 4
/ 8, float32 and bf16 autocast, every configuration runs the same sequences once to warm up (graph captures, cuDNN
algorithm choice), then ``reps`` timed passes, each ending in a device synchronise.  Also reported: the library's
kernel launches per batch with CUDA graphs off (``comet_launch_count``), and the graph captures of the coarse / fine
update transformers over 20 batches of 8 with freshly drawn counts.  One JSON object on stdout (and in --out)."""
import argparse
import contextlib
import json
import os
import random
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seqs", type=int, default=16)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--frames", type=int, default=16)
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this measurement needs a CUDA device"
    import comet_pose_estimation_b200 as cb
    from comet_pose_estimation_b200 import update_former_tc

    dev = torch.device("cuda")
    torch.manual_seed(0)
    tp = cb.TrackerPredictor().eval().to(dev)
    rng = random.Random(0)
    g = torch.Generator(device=dev).manual_seed(0)
    S, HW = args.frames, args.size
    counts = [rng.randint(256, 512) for _ in range(args.seqs)]
    images = [torch.randn(1, S, 3, HW, HW, device=dev, generator=g) for _ in counts]
    queries = [torch.rand(n, 2, device=dev, generator=g) * (HW - 1) for n in counts]

    def run_loop():
        for im, q in zip(images, queries):
            tp.track(im, q[None])

    def run_batched(bs):
        for k in range(0, len(counts), bs):
            tp.track_batch(torch.cat(images[k:k + bs]), queries[k:k + bs])

    def timed(fn):
        fn()                                          # warm-up: every shape of the timed passes
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.reps):
            fn()
        torch.cuda.synchronize()
        return args.reps * len(counts) / (time.perf_counter() - t0)

    result = {"device": torch.cuda.get_device_name(dev), "frames": S, "image": HW, "num_tracks": counts,
              "reps": args.reps, "sequences_per_s": {}}
    try:
        import subprocess

        result["power_limit"] = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                                                str(dev.index or 0)], capture_output=True, text=True).stdout.strip()
    except Exception:
        result["power_limit"] = "unknown"
    for prec in ("float32", "bf16_autocast"):
        ctx = (lambda: torch.autocast("cuda", dtype=torch.bfloat16)) if prec == "bf16_autocast" else contextlib.nullcontext
        row = {}
        with ctx():
            row["track_loop"] = timed(run_loop)
            for bs in (1, 2, 4, 8):
                row[f"track_batch_{bs}"] = timed(lambda: run_batched(bs))
        result["sequences_per_s"][prec] = row

    # library launches per call with eager transformer launches (graphs off)
    update_former_tc.USE_CUDA_GRAPH = False
    launches = {}
    with torch.no_grad():
        n0 = cb._lib.lib.comet_launch_count()
        tp.track(images[0], queries[0][None])
        launches["track_1_sequence"] = int(cb._lib.lib.comet_launch_count() - n0)
        for bs in (2, 4, 8):
            n0 = cb._lib.lib.comet_launch_count()
            tp.track_batch(torch.cat(images[:bs]), queries[:bs])
            launches[f"track_batch_{bs}"] = int(cb._lib.lib.comet_launch_count() - n0)
    update_former_tc.USE_CUDA_GRAPH = True
    result["library_launches_eager"] = launches

    # graph captures over 20 batches of 8 with fresh counts
    mods = {"coarse": tp.coarse_predictor.updateformer, "fine": tp.fine_predictor.updateformer}
    before = {k: getattr(m, "_tc_captures", 0) for k, m in mods.items()}
    for _ in range(20):
        qs = [torch.rand(rng.randint(256, 512), 2, device=dev, generator=g) * (HW - 1) for _ in range(8)]
        tp.track_batch(torch.cat(images[:8]), qs)
    torch.cuda.synchronize()
    result["ragged_graph_captures_20_batches_of_8"] = {k: getattr(m, "_tc_captures", 0) - before[k] for k, m in mods.items()}
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
