"""Sequences per second of ``TrackerPredictor.track_batch(..., clip_frames=...)`` on sliding windows of one video, against
the two ways of tracking those windows without it, on one GPU.

    python scripts/shared_frames_time.py [--reps 2] [--out profiles/shared_frames_time.json]

Workload: a seeded synthetic 512x512 video of 136 frames (428 MB of float32 pixels, larger than the 126 MB L2) cut
into 16 windows of 16 frames at stride 8, so every inner frame is in two windows.  Window w gets N_w tracks, N_w seeded
from U[256, 512], with query points in U[16, 496)^2 on its first frame.  Default configuration weights, seeded (timing
does not depend on their values).  Arms, each in float32 and under bf16 autocast:
  * ``clip_frames``: ``track_batch(video, ..., clip_frames=...)`` over batches of 8 windows;
  * ``gathered_copies``: ``track_batch`` over batches of 8 windows gathered into copies (the gather is timed: it is what
    a caller without ``clip_frames`` pays);
  * ``track_loop``: one ``track()`` per window.
Every arm runs once to warm up (graph captures, cuDNN algorithm choice); then ``reps`` rounds, each one timed pass of
every arm in turn, so the arms alternate.  A pass starts and ends with a device synchronise.  Reported per arm: sequences
per second over all timed passes, every pass time, the frames ``BasicEncoder`` encodes per pass (forward hook), the peak
device memory of its passes, and the update-transformer graph captures during its timed passes; with the card's name and
power limit read in the same run.  One JSON object on stdout (and in --out)."""
import argparse
import contextlib
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--windows", type=int, default=16)
    ap.add_argument("--length", type=int, default=16)
    ap.add_argument("--stride", type=int, default=8)
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this measurement needs a CUDA device"
    import comet_pose_estimation_b200 as cb

    dev = torch.device("cuda")
    torch.manual_seed(0)
    tp = cb.TrackerPredictor().eval().to(dev)
    HW, L, K, Wn = args.size, args.length, args.stride, args.windows
    T = (Wn - 1) * K + L
    g = torch.Generator(device=dev).manual_seed(0)
    video = torch.randn(T, 3, HW, HW, device=dev, generator=g)
    gen = torch.Generator().manual_seed(0)
    counts = torch.randint(256, 513, (Wn,), generator=gen).tolist()
    queries = [(torch.rand(n, 2, generator=gen) * (HW - 32) + 16).to(dev) for n in counts]
    windows = [list(range(w * K, w * K + L)) for w in range(Wn)]
    batches = [range(i, min(i + args.batch, Wn)) for i in range(0, Wn, args.batch)]

    encoded = [0]
    tp.coarse_fnet.register_forward_hook(lambda mod, inp, out: encoded.__setitem__(0, encoded[0] + inp[0].shape[0]))
    mods = {"coarse": tp.coarse_predictor.updateformer, "fine": tp.fine_predictor.updateformer}

    def captures():
        return sum(getattr(m, "_tc_captures", 0) for m in mods.values())

    def gathered(ws):
        return [video[windows[w][0]:windows[w][-1] + 1].clone() for w in ws]

    arms = {
        "clip_frames": lambda: [tp.track_batch(video, [queries[w] for w in ws], clip_frames=[windows[w] for w in ws])
                                for ws in batches],
        "gathered_copies": lambda: [tp.track_batch(gathered(ws), [queries[w] for w in ws]) for ws in batches],
        "track_loop": lambda: [tp.track(video[windows[w][0]:windows[w][-1] + 1][None], queries[w][None])
                               for w in range(Wn)],
    }
    power = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(dev.index or 0)],
                           capture_output=True, text=True).stdout.strip()
    result = {"device": torch.cuda.get_device_name(dev), "nvidia_smi_name_power_limit": power, "image": HW,
              "video_frames": T, "windows": Wn, "window_length": L, "stride": K, "batch": args.batch,
              "tracks_per_window": counts, "reps": args.reps, "results": {}}
    for prec in ("float32", "bf16_autocast"):
        ctx = torch.autocast("cuda", dtype=torch.bfloat16) if prec == "bf16_autocast" else contextlib.nullcontext()
        rows = {name: {"pass_s": [], "encoder_frames_per_pass": 0, "peak_memory_bytes": 0,
                       "graph_captures_in_timed_passes": 0} for name in arms}
        with ctx:
            for fn in arms.values():
                fn()
            torch.cuda.synchronize()
            for _ in range(args.reps):
                for name, fn in arms.items():
                    row = rows[name]
                    torch.cuda.reset_peak_memory_stats(dev)
                    c0, encoded[0] = captures(), 0
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    fn()
                    torch.cuda.synchronize()
                    row["pass_s"].append(time.perf_counter() - t0)
                    row["encoder_frames_per_pass"] = encoded[0]
                    row["peak_memory_bytes"] = max(row["peak_memory_bytes"], torch.cuda.max_memory_allocated(dev))
                    row["graph_captures_in_timed_passes"] += captures() - c0
        for row in rows.values():
            row["sequences_per_s"] = len(row["pass_s"]) * Wn / sum(row["pass_s"])
        result["results"][prec] = rows
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
