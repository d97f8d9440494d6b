"""Sequences per second of ``TrackerPredictor.track_batch(..., query_frames=...)`` against the two ways of tracking points
that start on later frames without it, on one GPU.

    python scripts/query_frames_time.py [--seqs 4] [--reps 2] [--out result.json]

Workload: ``seqs`` seeded 16-frame 512x512 sequences with 512 tracks each, spread evenly over G = 1, 2, 4, 8 query frames
(frames 0, 2, 4, ... of the sequence); seeded random images, default configuration weights (timing does not depend on
their values).  Arms, each in float32 and under bf16 autocast:
  * ``query_frames``: one ``track_batch`` over all sequences with ``query_frames``;
  * ``swapped_copies``: one ``track_batch`` over seqs * G copies of the images, each with frames 0 and q swapped and the
    tracks of query frame q (VGGSfM's switch_tensor_order, batched);
  * ``track_loop``: one ``track()`` per (sequence, query frame) on its swapped copy.
Every arm runs once to warm up (graph captures, cuDNN algorithm choice), then ``reps`` timed passes ending in a device
synchronise.  Reported per arm: sequences per second, the frames ``BasicEncoder`` encodes per pass (forward hook), and the
update-transformer graph captures during the timed passes.  One JSON object on stdout (and in --out)."""
import argparse
import contextlib
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def swap(x, q):
    order = list(range(x.shape[0]))
    order[0], order[q] = q, 0
    return x[order]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seqs", type=int, default=4)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--frames", type=int, default=16)
    ap.add_argument("--tracks", type=int, default=512)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this measurement needs a CUDA device"
    import comet_pose_estimation_b200 as cb

    dev = torch.device("cuda")
    torch.manual_seed(0)
    tp = cb.TrackerPredictor().eval().to(dev)
    g = torch.Generator(device=dev).manual_seed(0)
    HW, S, N, B = args.size, args.frames, args.tracks, args.seqs
    images = torch.randn(B, S, 3, HW, HW, device=dev, generator=g)
    queries = torch.rand(B, N, 2, device=dev, generator=g) * (HW - 1)

    encoded = [0]
    tp.coarse_fnet.register_forward_hook(lambda mod, inp, out: encoded.__setitem__(0, encoded[0] + inp[0].shape[0]))
    mods = {"coarse": tp.coarse_predictor.updateformer, "fine": tp.fine_predictor.updateformer}

    def captures():
        return sum(getattr(m, "_tc_captures", 0) for m in mods.values())

    power = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(dev.index or 0)],
                           capture_output=True, text=True).stdout.strip()
    result = {"device": torch.cuda.get_device_name(dev), "nvidia_smi_name_power_limit": power, "image": HW, "frames": S,
              "tracks_per_sequence": N, "sequences": B, "reps": args.reps, "results": {}}
    for G in (1, 2, 4, 8):
        qframes = [2 * k for k in range(G)]                          # query frames 0, 2, 4, ...
        qf = torch.tensor([qframes[n * G // N] for n in range(N)]).repeat(B, 1)        # (B, N), G equal groups
        groups = [(b, q, torch.nonzero(qf[b] == q)[:, 0].to(dev)) for b in range(B) for q in qframes]
        copies = torch.stack([swap(images[b], q) for b, q, _ in groups])
        copy_queries = [queries[b, sel] for b, _, sel in groups]

        arms = {
            "query_frames": lambda: tp.track_batch(images, queries, query_frames=qf),
            "swapped_copies": lambda: tp.track_batch(copies, copy_queries),
            "track_loop": lambda: [tp.track(copies[i:i + 1], copy_queries[i][None]) for i in range(len(groups))],
        }
        for prec in ("float32", "bf16_autocast"):
            ctx = torch.autocast("cuda", dtype=torch.bfloat16) if prec == "bf16_autocast" else contextlib.nullcontext()
            row = {}
            with ctx:
                for name, fn in arms.items():
                    fn()
                    torch.cuda.synchronize()
                    c0, encoded[0] = captures(), 0
                    t0 = time.perf_counter()
                    for _ in range(args.reps):
                        fn()
                    torch.cuda.synchronize()
                    dt = time.perf_counter() - t0
                    row[name] = {"sequences_per_s": args.reps * B / dt, "encoder_frames_per_pass": encoded[0] // args.reps,
                                 "graph_captures_in_timed_passes": captures() - c0}
            result["results"].setdefault(f"G{G}", {})[prec] = row
        del copies
        torch.cuda.empty_cache()
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
