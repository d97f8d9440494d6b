"""Sequences per second of ``TrackerPredictor.track_batch(..., num_frames=...)`` on sequences of different lengths, against
a loop of ``track()`` and against grouping the sequences by length, on one GPU.

    python scripts/ragged_frames_time.py [--seqs 16] [--reps 2] [--out result.json]

Workload: 16 seeded 512x512 sequences, S_b drawn from a seeded U{8..16} and N_b from U[256, 512]; seeded random images,
default configuration weights (timing does not depend on their values).  Arms, each in float32 and under bf16 autocast:
a loop of ``track()``; ``track_batch`` per group of equal S_b (in batches of at most 8: what a caller without
``num_frames`` must do); one ``track_batch`` with ``num_frames`` per batch of 1 / 2 / 4 / 8 sequences in input order.
Every arm runs once to warm up (graph captures, cuDNN algorithm choice), then ``reps`` timed passes ending in a device
synchronise; the update-transformer graph captures during the timed passes of each arm are reported beside it (the
transformers keep four graphs each, keyed by shape, so arms that see many shapes re-capture).  Also reported:
``num_frames=[16] * 8`` against ``num_frames=None`` on the same 8 sixteen-frame sequences (the cost of the frame-count
path without padding), ``--pad-reps`` passes of each, alternated, as per-pass milliseconds (median, min, max); the graph
captures over 20 batches of 8 with fresh counts; and the library's kernel launches per batch with CUDA graphs off
(``comet_launch_count``).  One JSON object on stdout (and in --out)."""
import argparse
import contextlib
import json
import os
import random
import statistics
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seqs", type=int, default=16)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--pad-reps", type=int, default=15)
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
    HW, SMAX = args.size, 16
    frames = [rng.randint(8, SMAX) for _ in range(args.seqs)]
    counts = [rng.randint(256, 512) for _ in range(args.seqs)]
    clips = [torch.randn(s, 3, HW, HW, device=dev, generator=g) for s in frames]
    queries = [torch.rand(n, 2, device=dev, generator=g) * (HW - 1) for n in counts]
    by_len = {}
    for i, s in enumerate(frames):
        by_len.setdefault(s, []).append(i)

    def run_loop():
        for c, q in zip(clips, queries):
            tp.track(c[None], q[None])

    def run_grouped():
        for idx in by_len.values():
            for k in range(0, len(idx), 8):
                part = idx[k:k + 8]
                tp.track_batch(torch.stack([clips[i] for i in part]), [queries[i] for i in part])

    def run_frames(bs):
        for k in range(0, len(clips), bs):
            tp.track_batch(clips[k:k + bs], queries[k:k + bs])

    mods = {"coarse": tp.coarse_predictor.updateformer, "fine": tp.fine_predictor.updateformer}

    def captures():
        return sum(getattr(m, "_tc_captures", 0) for m in mods.values())

    def timed(fn, n_seqs, name, row, caps):
        fn()
        torch.cuda.synchronize()
        c0 = captures()
        t0 = time.perf_counter()
        for _ in range(args.reps):
            fn()
        torch.cuda.synchronize()
        row[name] = args.reps * n_seqs / (time.perf_counter() - t0)
        caps[name] = captures() - c0

    power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", str(dev.index or 0)],
                           capture_output=True, text=True).stdout.strip()
    result = {"device": torch.cuda.get_device_name(dev), "power_limit": power, "image": HW, "num_frames": frames,
              "num_tracks": counts, "reps": args.reps, "sequences_per_s": {}}
    full = [torch.randn(SMAX, 3, HW, HW, device=dev, generator=g) for _ in range(8)]
    full_b = torch.stack(full)
    for prec in ("float32", "bf16_autocast"):
        ctx = (lambda: torch.autocast("cuda", dtype=torch.bfloat16)) if prec == "bf16_autocast" else contextlib.nullcontext
        row, caps = {}, {}
        with ctx():
            timed(run_loop, len(clips), "track_loop", row, caps)
            timed(run_grouped, len(clips), "track_batch_grouped_by_length", row, caps)
            for bs in (1, 2, 4, 8):
                timed(lambda: run_frames(bs), len(clips), f"track_batch_num_frames_{bs}", row, caps)
            # no padding: the frame-count path against the plain one, alternated pass by pass
            t = {"None": [], "16": []}
            for kw in ({}, {"num_frames": [SMAX] * 8}):
                tp.track_batch(full_b, queries[:8], **kw)
            for _ in range(args.pad_reps):
                for name, kw in (("None", {}), ("16", {"num_frames": [SMAX] * 8})):
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    tp.track_batch(full_b, queries[:8], **kw)
                    torch.cuda.synchronize()
                    t[name].append(1e3 * (time.perf_counter() - t0))
            result.setdefault("batch_8_16_frames_ms_per_pass", {})[prec] = {
                f"num_frames_{k}": {"median": statistics.median(v), "min": min(v), "max": max(v), "passes": len(v)}
                for k, v in t.items()}
        result["sequences_per_s"][prec] = row
        result.setdefault("graph_captures_in_timed_passes", {})[prec] = caps

    before = {k: getattr(m, "_tc_captures", 0) for k, m in mods.items()}
    for _ in range(20):
        fs = [rng.randint(8, SMAX) for _ in range(8)]
        qs = [torch.rand(rng.randint(256, 512), 2, device=dev, generator=g) * (HW - 1) for _ in range(8)]
        tp.track_batch(full_b, qs, num_frames=fs)
    torch.cuda.synchronize()
    result["graph_captures_20_batches_of_8_fresh_counts"] = {k: getattr(m, "_tc_captures", 0) - before[k]
                                                             for k, m in mods.items()}

    update_former_tc.USE_CUDA_GRAPH = False
    launches = {}
    with torch.no_grad():
        n0 = cb._lib.lib.comet_launch_count()
        tp.track(clips[0][None], queries[0][None])
        launches["track_1_sequence"] = int(cb._lib.lib.comet_launch_count() - n0)
        for bs in (2, 4, 8):
            n0 = cb._lib.lib.comet_launch_count()
            tp.track_batch(clips[:bs], queries[:bs])
            launches[f"track_batch_num_frames_{bs}"] = int(cb._lib.lib.comet_launch_count() - n0)
    update_former_tc.USE_CUDA_GRAPH = True
    result["library_launches_eager"] = launches
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
