"""Sequences per second of ``TrackerPredictor.track_batch`` over sequences of different image sizes against the two ways
of tracking them without it, on one GPU.

    python scripts/image_sizes_time.py [--seqs 16] [--batch 8] [--reps 3] [--out result.json]

Workload: ``seqs`` seeded 16-frame sequences, each of a size drawn from {384x384, 512x512, 480x640, 640x480} and with
256-512 tracks (seeded); seeded random images, default configuration weights (timing does not depend on their values).
Arms, each in float32 and under bf16 autocast:
  * ``mixed``: one ``track_batch`` per ``batch`` sequences, sizes mixed (a list of clips);
  * ``per_size``: one ``track_batch`` per size group (all sequences of one size);
  * ``track_loop``: one ``track()`` per sequence.
Every arm runs once to warm up every shape it uses (graph captures, cuDNN algorithm choice), then ``reps`` timed passes,
each ending in a device synchronise; the time of every pass is reported to show the spread.  Per arm also: the peak
device memory of the timed passes (``torch.cuda.max_memory_allocated``, the images included) and the update-transformer
graph captures during them.  The packed frame buffer's size is reported beside what a copy padded to the largest size
would take.  One JSON object on stdout (and in --out)."""
import argparse
import contextlib
import json
import os
import random
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

SIZES = [(384, 384), (512, 512), (480, 640), (640, 480)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seqs", type=int, default=16)
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--frames", type=int, default=16)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this measurement needs a CUDA device"
    import comet_pose_estimation_b200 as cb

    dev = torch.device("cuda")
    torch.manual_seed(0)
    tp = cb.TrackerPredictor().eval().to(dev)
    rng = random.Random(0)
    g = torch.Generator(device=dev).manual_seed(0)
    B, S = args.seqs, args.frames
    sizes = [rng.choice(SIZES) for _ in range(B)]
    counts = [rng.randint(256, 512) for _ in range(B)]
    clips = [torch.randn(S, 3, h, w, device=dev, generator=g) for h, w in sizes]
    queries = [torch.rand(n, 2, device=dev, generator=g) * torch.tensor([w - 1.0, h - 1.0], device=dev)
               for n, (h, w) in zip(counts, sizes)]
    by_size = {}
    for b, hw in enumerate(sizes):
        by_size.setdefault(hw, []).append(b)

    mods = {"coarse": tp.coarse_predictor.updateformer, "fine": tp.fine_predictor.updateformer}

    def captures():
        return sum(getattr(m, "_tc_captures", 0) for m in mods.values())

    arms = {
        "mixed": lambda: [tp.track_batch(clips[i:i + args.batch], queries[i:i + args.batch])
                          for i in range(0, B, args.batch)],
        "per_size": lambda: [tp.track_batch([clips[b] for b in bs], [queries[b] for b in bs]) for bs in by_size.values()],
        "track_loop": lambda: [tp.track(clips[b][None], queries[b][None]) for b in range(B)],
    }
    power = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(dev.index or 0)],
                           capture_output=True, text=True).stdout.strip()
    packed_elems = sum(c.numel() for c in clips)
    hmax, wmax = max(h for h, _ in sizes), max(w for _, w in sizes)
    result = {"device": torch.cuda.get_device_name(dev), "nvidia_smi_name_power_limit": power, "frames": S,
              "sequences": B, "batch": args.batch, "reps": args.reps,
              "sizes": [f"{h}x{w}" for h, w in sizes], "tracks": counts,
              "packed_buffer_mb": packed_elems * 4 / 2 ** 20, "padded_copy_mb": B * S * 3 * hmax * wmax * 4 / 2 ** 20,
              "results": {}}
    for prec in ("float32", "bf16_autocast"):
        ctx = torch.autocast("cuda", dtype=torch.bfloat16) if prec == "bf16_autocast" else contextlib.nullcontext()
        row = {}
        with ctx:
            for name, fn in arms.items():
                fn()
                torch.cuda.synchronize()
                torch.cuda.reset_peak_memory_stats(dev)
                c0 = captures()
                passes = []
                for _ in range(args.reps):
                    t0 = time.perf_counter()
                    fn()
                    torch.cuda.synchronize()
                    passes.append(time.perf_counter() - t0)
                row[name] = {"sequences_per_s": args.reps * B / sum(passes), "pass_s": passes,
                             "peak_memory_mb": torch.cuda.max_memory_allocated(dev) / 2 ** 20,
                             "graph_captures_in_timed_passes": captures() - c0}
        result["results"][prec] = row
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
