#!/usr/bin/env python
"""Benchmark of the COMET tracking hot path on B200 (contract: see the task statement / DESIGN.md section 6).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch Q] [--impl ours|reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1], "batched inference, seqlen=16, synthetic sequences on 1xB200"): one *step*
is one pass of the hot path over a batch of Q synthetic 16-frame sequences per GPU.  Per sequence that is
exactly what COMET.forward_all makes the tracker's correlation / lookup / token code do:

  coarse tracker  fmaps (1,16,128,64,64), N=512 tracks, L=5, r=4:  pyramid + pos-emb once, then 4 iterations of
                  [correlation -> 9x9x5 window lookup -> track tokens (1,512,16,664)]
  fine tracker    patch features (512,16,32,31,31), 1 track/patch, L=3, r=3: pyramid + pos-emb once, then
                  6 iterations of [correlation -> 7x7x3 lookup -> tokens (512,1,16,216)].  The patch features are the
                  2x-1 bilinear up-sampling of the patch encoder's 16x16 output (blocks.py:176-190); the default
                  --fine-layout up2 hands the path that 16x16 map, as this package's refine_track does (the up-sampled
                  tensor is never materialised); cl / nchw hand it the materialised 31x31 tensor (variants).

The update transformer that runs between iterations is outside the path (SURVEY 8f), so every iteration reads its
own pre-generated coords / track_feats (seeded random walk around the query points) -- the bytes and flops of the
path are exactly those of the real loop.  metric = sequences/s (whole job, all GPUs).

  value  inputs already resident in HBM when the timed region starts
  e2e    same pass through the public Python API with HOST (pinned) buffers: H2D of every input and D2H of the
         last-iteration tokens inside the timed region
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

COARSE = dict(S=16, N=512, C=128, H=64, W=64, L=5, r=4, iters=4, fine=False)
FINE = dict(S=16, P=512, C=32, H=31, W=31, L=3, r=3, iters=6, fine=True)
METRIC = "sequences/sec (seqlen=16)"
UNIT = "sequences/s"
DUMP_BYTES = 63 * 10 ** 6      # data of all --dump-outputs arrays together: under 64 MB with the .npy headers


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def tdim(L, r, latent, fine):
    d = L * (2 * r + 1) ** 2 + 2 * latent
    if fine:
        d += 4 if d % 2 == 0 else 5
    else:
        d += (4 - d % 4) % 4
    return d


# --------------------------------------------------------------------------- synthetic inputs (host, seeded)
def upsample_fine(torch, src, layout):
    """The fine tracker's materialised patch features: F.interpolate(src, 31x31, bilinear, align_corners=True) -- what
    ShallowEncoder.forward returns (blocks.py:176-190) -- as a channels-last view ("cl") or NCHW-contiguous ("nchw")."""
    import torch.nn.functional as F

    B, S, C, hs, ws = src.shape
    H, W = 2 * hs - 1, 2 * ws - 1
    out = torch.empty(B, S, H, W, C, dtype=torch.float32, device=src.device).permute(0, 1, 4, 2, 3)
    step = max(1, 4096 // S)
    for b0 in range(0, B, step):
        x = src[b0:b0 + step]
        out[b0:b0 + step] = F.interpolate(x.reshape(-1, C, hs, ws), (H, W), mode="bilinear",
                                          align_corners=True).reshape(x.shape[0], S, C, H, W)
    return out if layout == "cl" else out.contiguous()


def make_inputs(Q, seed, torch, pin, fine_layout="up2"):
    """Host tensors for Q sequences.  SURVEY 8(d) item 5: fmaps ~ N(0,1); queries U over the map; per-iteration
    coords = query + small random walk (frame 0 pinned); per-iteration track_feats ~ N(0,1).  The fine tracker's
    input is generated as the patch encoder's 16x16 output ~ N(0,1) (channels-last memory); for the cl / nchw layouts
    it is up-sampled to 31x31 here (outside any timed region), so every layout carries the same values."""
    g = torch.Generator().manual_seed(seed)

    def alloc(*shape):
        t = torch.empty(*shape, dtype=torch.float32)
        return t.pin_memory() if pin else t

    out = {}
    for name, cfg, B, N in (("coarse", COARSE, Q, COARSE["N"]), ("fine", FINE, Q * FINE["P"], 1)):
        S, C, H, W, it = cfg["S"], cfg["C"], cfg["H"], cfg["W"], cfg["iters"]
        if name == "fine":
            hs, ws = H // 2 + 1, W // 2 + 1
            src = torch.empty(B, S, hs, ws, C, dtype=torch.float32).permute(0, 1, 4, 2, 3)   # channels-last memory
            src.normal_(generator=g)
            if fine_layout == "up2":
                fm = alloc(B, S, hs, ws, C).permute(0, 1, 4, 2, 3)
                fm.copy_(src)
            else:
                up = upsample_fine(torch, src, fine_layout)
                fm = (alloc(B, S, H, W, C).permute(0, 1, 4, 2, 3) if fine_layout == "cl" else alloc(B, S, C, H, W))
                fm.copy_(up)
                del up
            del src
        else:
            fm = alloc(B, S, C, H, W)
            fm.normal_(generator=g)
        q = torch.rand(B, 1, N, 2, generator=g) * torch.tensor([W - 1.0, H - 1.0])
        coords = alloc(it, B, S, N, 2)
        feats = alloc(it, B, S, N, C)
        feats.normal_(generator=g)
        walk = torch.zeros(B, S, N, 2)
        for i in range(it):
            walk = walk + torch.randn(B, S, N, 2, generator=g) * 0.75
            c = q + walk
            c[:, 0] = q[:, 0]
            coords[i].copy_(c)
        out[name] = dict(fmaps=fm, coords=coords, feats=feats)
    return out


# --------------------------------------------------------------------------- our arm
class HotPath:
    """The hot path of one batch through the public API of comet_pose_estimation_b200."""

    def __init__(self, cb, torch, Q, dev):
        self.cb, self.torch, self.Q, self.dev = cb, torch, Q, dev
        self.td_c = tdim(COARSE["L"], COARSE["r"], COARSE["C"], False)
        self.td_f = tdim(FINE["L"], FINE["r"], FINE["C"], True)
        self.tok_c = torch.empty(Q, COARSE["N"], COARSE["S"], self.td_c, device=dev)
        self.tok_f = torch.empty(Q * FINE["P"], 1, FINE["S"], self.td_f, device=dev)
        self.events = None  # optional per-kernel timing

    def _mark(self, tag):
        if self.events is not None:
            e = self.torch.cuda.Event(enable_timing=True)
            e.record()
            self.events.append((tag, e))

    def run(self, d):
        cb = self.cb
        for name, cfg, out in (("coarse", COARSE, self.tok_c), ("fine", FINE, self.tok_f)):
            x = d[name]
            self._mark(None)
            if name == "fine" and x["fmaps"].shape[-1] != cfg["W"]:      # the encoder's half-resolution map (up2)
                blk = cb.CorrBlock.from_upsampled(x["fmaps"], num_levels=cfg["L"], radius=cfg["r"])
            else:
                blk = cb.CorrBlock(x["fmaps"], num_levels=cfg["L"], radius=cfg["r"])
            self._mark(name + "_pyramid")
            tk = cb.TrackTokenizer(blk, x["coords"][0][:, 0], out.shape[-1])
            self._mark(name + "_posemb")
            for i in range(cfg["iters"]):
                tk.tokens(x["coords"][i], x["feats"][i], out=out)
                self._mark(name + "_tokens")
        return self.tok_c, self.tok_f


def sample_outputs(outputs, budget=DUMP_BYTES):
    """Host float32 copies of `outputs` (name -> tensor), DUMP_BYTES in all.  A tensor larger than its share of the
    budget is cut to a fixed, seeded sample of rows (leading axes flattened, last axis whole, rows in order), so two
    runs with the same arguments keep the same elements."""
    import numpy as np
    import torch

    share = budget // len(outputs)
    out = {}
    for name, t in outputs.items():
        if t.numel() * 4 > share:
            rows = t.reshape(-1, t.shape[-1])
            keep = np.sort(np.random.default_rng(0).choice(rows.shape[0], share // (rows.shape[1] * 4), replace=False))
            t = rows[torch.as_tensor(keep, device=rows.device)]
        out[name] = t.float().cpu().numpy()
    return out


def fine_lines_per_query(coords, layout):
    """Mean number of 128-byte feature lines one fine query must read, from the ACTUAL coordinates: every box of the
    lookup is clipped to its map (taps off the map are zero padding and cost no traffic -- the TMA unit zero-fills them
    without fetching).  coords: (..., 2) float tensor in level-0 (31x31) cell units."""
    f = FINE
    x, y = coords[..., 0].double(), coords[..., 1].double()

    def inmap(c, scale, r, edge, size):
        o = (c * scale).floor() - r
        return ((o + edge).clamp(max=size) - o.clamp(min=0)).clamp(min=0)

    r = f["r"]
    if layout == "up2":
        hs = f["H"] // 2 + 1
        h2 = (hs - 1) // 2
        n = inmap(x, 0.5, r, 9, hs) * inmap(y, 0.5, r, 9, hs) + inmap(x, 0.25, r, 8, h2) * inmap(y, 0.25, r, 8, h2)
    else:
        n, h = 0, f["H"]
        for l in range(f["L"]):
            n = n + inmap(x, 0.5 ** l, r, 2 * r + 2, h) * inmap(y, 0.5 ** l, r, 2 * r + 2, h)
            h //= 2
    return float(n.mean())


def algorithmic_bytes(Q, fine_coords=None, fine_layout="up2"):
    """DESIGN.md section 5: bytes one launch has to move.  fine_tokens uses the window-neighbourhood definition (SURVEY
    8d) with every box clipped to its map per query (round-1's figure counted taps the hardware never fetches)."""
    c, f = COARSE, FINE
    tdc, tdf = tdim(c["L"], c["r"], c["C"], False), tdim(f["L"], f["r"], f["C"], True)
    # coarse: SURVEY 8(d) compulsory traffic (whole level-0 map + targets + coords + tokens)
    coarse = Q * (c["S"] * c["C"] * c["H"] * c["W"] * 4 + c["S"] * c["N"] * c["C"] * 4 + c["S"] * c["N"] * 8
                  + c["N"] * c["S"] * tdc * 4)
    if fine_coords is not None:
        lines = fine_lines_per_query(fine_coords, fine_layout)
    elif fine_layout == "up2":
        hs = f["H"] // 2 + 1
        lines = min(9, hs) ** 2 + min(2 * f["r"] + 2, (hs - 1) // 2) ** 2      # S box + level-2 box, unclipped by position
    else:
        G = 2 * f["r"] + 2
        lines, h = 0, f["H"]
        for _ in range(f["L"]):
            lines += min(G, h) ** 2
            h //= 2
    per_q = lines * f["C"] * 4 + f["C"] * 4 + 8 + tdf * 4 + tdf * 4 / f["S"]
    fine = Q * f["P"] * f["S"] * per_q
    pyr_c = Q * c["S"] * c["C"] * 4 * (64 * 64 + 2 * (32 * 32 + 16 * 16 + 8 * 8) + 4 * 4)
    if fine_layout == "up2":
        hs = f["H"] // 2 + 1
        # read the 15x15 positions of the 16x16 source that level 2 depends on, write level 2
        pyr_f = Q * f["P"] * f["S"] * f["C"] * 4 * ((hs - 1) ** 2 + ((hs - 1) // 2) ** 2)
    else:
        # read the 30x30 positions of level 0 that floor-mode pooling uses, write levels 1-2
        pyr_f = Q * f["P"] * f["S"] * f["C"] * 4 * (30 * 30 + 15 * 15 + 7 * 7)
    return dict(coarse_tokens=coarse, fine_tokens=fine, coarse_pyramid=pyr_c, fine_pyramid=pyr_f,
                fine_lines_per_query=lines)


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "20"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            txt = self.p.communicate(timeout=5)[0]
        except Exception:
            self.p.kill()
            txt = ""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in txt.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------- CPU baseline (oracle port)
def cpu_hot_path(torch, d):
    """One pass of the SAME hot path on the host cores through oracle/torch_port.py (the reference's own ATen calls):
    per sequence coarse 4 iterations + fine 6 iterations, pyramids included.  The fine tracker gets the materialised
    31x31 patch features (what the reference's CorrBlock receives)."""
    from oracle import torch_port as P

    with torch.no_grad():
        for name, cfg in (("coarse", COARSE), ("fine", FINE)):
            x = d[name]
            td = tdim(cfg["L"], cfg["r"], cfg["C"], cfg["fine"])
            lv = P.pyramid(x["fmaps"], cfg["L"])
            for i in range(cfg["iters"]):
                P.hot_path_iteration(lv, x["coords"][i], x["feats"][i], cfg["r"], (cfg["H"], cfg["W"]), td)


def cpu_reference_seq_per_s(torch, reps):
    """cpu_baseline of the GPU arm's line: ONE sequence per rep (bounded sample), best of `reps` after a warm-up."""
    ncores = os.cpu_count() or 1
    torch.set_num_threads(ncores)
    d = make_inputs(1, 1234, torch, pin=False, fine_layout="nchw")
    times = []
    for rep in range(reps + 1):
        t0 = time.perf_counter()
        cpu_hot_path(torch, d)
        dt = time.perf_counter() - t0
        if rep > 0 or reps == 0:
            times.append(dt)
    return 1.0 / min(times), statistics.mean(times), ncores


TRACKER = dict(coarse=dict(stride=4, corr_levels=5, corr_radius=4, latent_dim=128, hidden_size=384, depth=6, use_spaceatt=True, fine=False),
               fine=dict(stride=1, corr_levels=3, corr_radius=3, latent_dim=32, hidden_size=256, depth=4, use_spaceatt=False, fine=True))


def cpu_encoders_s(torch):
    """CPU baseline scope (iii) of BASELINE.md section 4, the part scope (ii) does not contain: the two encoders of one
    sequence on the host cores -- BasicEncoder on 16 frames of 512x512 and ShallowEncoder on 512 x 16 patches of 31x31
    (their torch.nn / ATen definition, which is what the reference executes; random-init weights, one pass each after a
    small warm-up; the patch encoder runs in chunks of 1024 patches like refine_track does for memory)."""
    import importlib

    tp = importlib.import_module("comet_pose_estimation_b200.track_predictor")
    rt = importlib.import_module("comet_pose_estimation_b200.refine_track")
    torch.manual_seed(0)
    basic, shallow = tp.BasicEncoder().eval(), rt.ShallowEncoder().eval()
    frames = torch.randn(16, 3, 512, 512)
    patches = torch.randn(COARSE["N"] * 16, 3, 31, 31)
    with torch.no_grad():
        basic(frames[:1]); shallow(patches[:64])          # warm-up (thread pool, oneDNN primitives)
        t0 = time.perf_counter()
        basic(frames)
        t1 = time.perf_counter()
        for i in range(0, patches.shape[0], 1024):
            shallow(patches[i:i + 1024])
        t2 = time.perf_counter()
    return t1 - t0, t2 - t1


def cpu_tracker_loop_s(torch, reps=1):
    """CPU baseline scope (ii) of BASELINE.md section 4: coarse (4 it) + fine (6 it) tracker loops of ONE sequence WITH the
    update transformer -- hot path through oracle/torch_port.py (the reference's ATen calls), transformer and state update
    through torch.nn on the host cores (the same module definition the reference uses, update_former._forward_torch)."""
    from oracle import torch_port as P
    import importlib

    uf = importlib.import_module("comet_pose_estimation_b200.update_former")
    torch.manual_seed(0)
    d = make_inputs(1, 4321, torch, pin=False, fine_layout="nchw")
    mods = {}
    for name, cfg in (("coarse", COARSE), ("fine", FINE)):
        t = TRACKER[name]
        td = tdim(cfg["L"], cfg["r"], cfg["C"], cfg["fine"])
        mods[name] = (uf.EfficientUpdateFormer(space_depth=t["depth"] if t["use_spaceatt"] else 0, time_depth=t["depth"], input_dim=td,
                                               hidden_size=t["hidden_size"], output_dim=t["latent_dim"] + 2,
                                               add_space_attn=t["use_spaceatt"]).eval(),
                      torch.nn.GroupNorm(1, t["latent_dim"]), torch.nn.Sequential(torch.nn.Linear(t["latent_dim"], t["latent_dim"]), torch.nn.GELU()))
    best = None
    with torch.no_grad():
        for rep in range(reps + 1):
            t0 = time.perf_counter()
            for name, cfg in (("coarse", COARSE), ("fine", FINE)):
                x = d[name]
                former, norm, upd = mods[name]
                td = tdim(cfg["L"], cfg["r"], cfg["C"], cfg["fine"])
                lv = P.pyramid(x["fmaps"], cfg["L"])
                coords, feats = x["coords"][0].clone(), x["feats"][0].clone()
                B, S, N, C = feats.shape
                for _ in range(cfg["iters"]):
                    tok = P.hot_path_iteration(lv, coords, feats, cfg["r"], (cfg["H"], cfg["W"]), td)
                    delta = former._forward_torch(tok).reshape(B * N, S, C + 2)
                    f_ = feats.permute(0, 2, 1, 3).reshape(B * N * S, C)
                    f_ = upd(norm(delta[:, :, 2:].reshape(B * N * S, C))) + f_
                    feats = f_.reshape(B, N, S, C).permute(0, 2, 1, 3)
                    coords = coords + delta[:, :, :2].reshape(B, N, S, 2).permute(0, 2, 1, 3) * 0.01
            dt = time.perf_counter() - t0
            if rep > 0 or reps == 0:
                best = dt if best is None else min(best, dt)
    return best


def make_config(Q, world, fine_layout):
    """`config` of the JSON line -- identical in both arms (the workload, not the implementation)."""
    return {"workload": workload_name(Q), "sequences_per_gpu_per_step": Q, "seqlen": 16,
            "parallelism": f"dp{world} (sequences sharded across ranks, no collective)",
            "fine_input": "patch encoder output 16x16x32 per (track, frame); the fine tracker's 31x31 features are its "
                          "2x-1 bilinear up-sampling (blocks.py:176-190)",
            "l2": "inputs per step exceed L2 (fine patch features: %.1f GB at 31x31, %.2f GB at 16x16)"
                  % (Q * 1.008, Q * 0.268)}


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (pinned port, kind "port") on all host cores,
    SAME workload as the GPU arm: `--batch` sequences per step."""
    import torch

    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    t0 = time.perf_counter()
    ncores = os.cpu_count() or 1
    torch.set_num_threads(ncores)
    Q = args.batch
    d = make_inputs(Q, 1234, torch, pin=False, fine_layout="nchw")
    for _ in range(args.warmup):
        cpu_hot_path(torch, d)
    t1 = time.perf_counter()
    for _ in range(args.steps):
        cpu_hot_path(torch, d)
    el = time.perf_counter() - t1
    v = Q * args.steps / el
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * el / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": make_config(Q, max(1, args.gpus), args.fine_layout),
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": ncores, "kind": "port",
                         "sample": f"{Q} sequences/step (the GPU arm's batch): coarse 4 it + fine 6 it, pyramids included; "
                                   "oracle/torch_port.py (the reference's own ATen calls), torch CPU fp32, rank 0 only"},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": time.perf_counter() - t0,
    }
    print(json.dumps(line), flush=True)
    return 0


def workload_name(Q):
    return (f"COMET tracking hot path, batch of {Q} synthetic 16-frame sequences per GPU: coarse "
            f"(S=16,N=512,C=128,64x64,L=5,r=4,4 it) + fine (512 patches,S=16,C=32,31x31,L=3,r=3,6 it); "
            f"pyramid + pos-emb + fused corr/lookup/token kernels")


# --------------------------------------------------------------------------- main (our arm)
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=4, help="sequences per GPU per step")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-reps", type=int, default=30, help="CPU baseline: sequences timed after one warm-up (~0.27 s each)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-variants", action="store_true")
    ap.add_argument("--fine-layout", default="up2", choices=["up2", "cl", "nchw"],
                    help="what the fine tracker is handed: up2 = the patch encoder's 16x16 output (this package's "
                         "refine_track: the 31x31 up-sampling is evaluated inside the lookup); cl = materialised 31x31 "
                         "features as a channels-last view; nchw = contiguous (B,S,C,H,W) as the reference's own "
                         "refine_track would hand over")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the tokens the last timed step computed (rank 0) as "
                         "DIR/coarse_tokens.npy and DIR/fine_tokens.npy, float32; beyond 64 MB in all, a fixed seeded "
                         "sample of token rows is written")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    import torch

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback exists)"
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus or world == 1, f"--gpus {args.gpus} but WORLD_SIZE={world}"

    import comet_pose_estimation_b200 as cb
    from comet_pose_estimation_b200 import launch as cl

    # host buffers node-local to the GPU (matters for the end-to-end arm once several ranks copy at the same time)
    prev_affinity = cl.bind_to_gpu_numa_node(local) if world > 1 else None

    Q = args.batch
    layout = args.fine_layout
    host = make_inputs(Q, 1000 + rank, torch, pin=True, fine_layout=layout)
    # empty_like + copy_ keep the strides (a channels-last view stays a channels-last view on the device)
    devin = {k: {n: torch.empty_like(t, device=dev).copy_(t, non_blocking=True) for n, t in v.items()}
             for k, v in host.items()}
    torch.cuda.synchronize()
    hp = HotPath(cb, torch, Q, dev)

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if dist is None:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn, steps, warmup, per_class=False):
        """W warm-ups, barrier, K steps between two events on the launching stream, barrier; max over ranks."""
        for _ in range(warmup):
            fn()
        barrier()
        if per_class:
            hp.events = []
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ev, hp.events = hp.events, None
        per = {}
        if ev:
            for (t0_, a_), (t1_, b_) in zip(ev[:-1], ev[1:]):
                if t1_ is not None:
                    per.setdefault(t1_, []).append(a_.elapsed_time(b_))
        return max_over_ranks(e0.elapsed_time(e1)) / steps, per

    # ---- device-resident arm ------------------------------------------------------------------
    sampler = ClockSampler(local) if rank == 0 else None   # samples every 20 ms from the warm-up to the end of the timed region
    launches0 = None

    def step_dev():
        hp.run(devin)

    for _ in range(args.warmup):
        step_dev()
    barrier()
    launches0 = cb._lib.lib.comet_launch_count()
    ms_step, per = timed(step_dev, args.steps, 0, per_class=True)
    launches = cb._lib.lib.comet_launch_count() - launches0  # counted by the library itself, one per kernel launch
    clocks = sampler.stop() if sampler else None
    value = Q * world / (ms_step * 1e-3)
    if args.dump_outputs and rank == 0:
        # the variants below reuse hp's output buffers: save the timed step's tokens now
        import numpy as np

        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in sample_outputs({"coarse_tokens": hp.tok_c, "fine_tokens": hp.tok_f}).items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)

    kern = {k: {"launch_groups": len(v), "ms_avg": sum(v) / len(v), "ms_per_step": sum(v) / args.steps}
            for k, v in per.items()}
    ab = algorithmic_bytes(Q, host["fine"]["coords"], layout)
    dom = max(kern, key=lambda k: kern[k]["ms_per_step"])
    peak, peak_src = peaks()
    for k in kern:
        if k in ab:
            kern[k]["algorithmic_MB"] = ab[k] / 1e6
            kern[k]["GBps"] = ab[k] / (kern[k]["ms_avg"] * 1e-3) / 1e9
    # roofline of the dominant kernel class (by device time inside the timed region).  Every class of this path is
    # HBM-bound; `traffic` = dram__bytes_read.sum + dram__bytes_write.sum of ONE launch at this batch size and layout
    # from the committed ncu --set full captures (profiles/traffic.json, written by scripts/ncu_summary.py --traffic).
    KNAME = {
        "fine_tokens": {"up2": "corr_lookup_c32_up2_kernel<TOKENS> (fine tracker: TMA-staged corr + lookup + tokens on the 16x16 source map)",
                        "cl": "corr_lookup_c32_tma_kernel<R=3,TOKENS> (fine tracker: TMA-staged corr + lookup + tokens)",
                        "nchw": "corr_lookup_c32_kernel<R=3,TOKENS> (fine tracker: fused corr + lookup + tokens)"},
        "fine_pyramid": {"up2": "pyramid_up2_kernel (fine tracker: level 2 pooled straight from the 16x16 source map)",
                         "cl": "pyramid_cl_in_fine_kernel (fine tracker: channel-last pyramid)",
                         "nchw": "pyramid_cl_fine_kernel (fine tracker: NCHW -> channel-last pyramid)"},
        "coarse_tokens": {"cl": "tc_pre_kernel + corr_tc_kernel (coarse tracker: tcgen05 corr + lookup + tokens)"},
        "coarse_pyramid": {"cl": "tc_prepare_kernel (coarse pyramid + bf16 hi/lo split)"},
    }
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj_all = json.load(f)
    except Exception:
        tj_all = {}

    def roofline_of(cls):
        k = kern[cls]
        tj = tj_all.get(f"{cls}/{layout}") or (tj_all.get(cls) if not cls.startswith("fine") else None) or {}
        traffic = tj.get("dram_bytes_per_launch") if tj.get("batch") == Q else None
        names = KNAME.get(cls, {})
        gbps = k.get("GBps")
        return {"bound": "hbm", "kernel": names.get(layout, names.get("cl", cls)),
                "achieved": gbps, "peak": peak, "unit": "GB/s",
                "frac": (gbps / peak) if gbps else None, "traffic": traffic,
                "frac_dram": (traffic / (k["ms_avg"] * 1e-3) / 1e9 / peak) if traffic else None,
                "traffic_source": tj.get("source") if traffic else None, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": ab.get(cls), "ms_per_launch": k["ms_avg"]}

    roof = roofline_of(dom if dom in ab else "fine_tokens")
    roof["dominant_by_time"] = dom
    if dom == "coarse_tokens":
        # the coarse class is the tcgen05 correlation kernel: its roof is the tensor pipe (north_star), FLOPs as the
        # reference defines them (dense, all pyramid levels); the HBM view of the same launches stays in `rooflines`
        k_ = kern["coarse_tokens"]
        flop_ = 2.0 * Q * COARSE["S"] * COARSE["N"] * COARSE["C"] * 5456
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f_:
                tp_ = float(json.load(f_)["bf16_tflops_sustained"])
        except Exception:
            tp_ = 1400.0
        roof.update({"bound": "tensor", "achieved": flop_ / (k_["ms_avg"] * 1e-3) / 1e12, "peak": tp_, "unit": "TFLOP/s",
                     "frac": flop_ / (k_["ms_avg"] * 1e-3) / 1e12 / tp_, "frac_dram": None,
                     "algorithmic_flops_per_launch": flop_,
                     "peak_source": "measured (MEASURED_PEAKS.json, sustained bf16)"})
    roof["note"] = ("algorithmic bytes: fine_tokens = per query the feature lines of its boxes CLIPPED to the maps (from the "
                    "actual coordinates; %.1f lines of 128 B on average) + target + coords + token row; fine_pyramid = "
                    "the source positions level 2 depends on read once + level 2 written; coarse_tokens = SURVEY 8d "
                    "compulsory traffic (fp32 maps + targets + coords + tokens).  frac_dram = measured DRAM bytes "
                    "(ncu, profiles/traffic.json) / time / peak" % ab["fine_lines_per_query"])
    rooflines = {c: roofline_of(c) for c in kern if c in ab}
    # correlation on the tensor pipe (coarse tracker): FLOPs as the reference defines them (dense, all pyramid levels,
    # one pass).  The kernel issues 3 bf16 passes (fp32 parity) but only for the band of map rows each sorted query
    # tile touches (~45 % of the tiles at this query distribution).
    ct = kern["coarse_tokens"]
    flop_alg = 2.0 * Q * COARSE["S"] * COARSE["N"] * COARSE["C"] * 5456
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            tpeak = float(json.load(f)["bf16_tflops_sustained"])
    except Exception:
        tpeak = 1400.0
    tensor = {"bound": "tensor", "kernel": "corr_tc_kernel (coarse tracker: tcgen05 correlation + lookup + tokens)",
              "achieved": flop_alg / (ct["ms_avg"] * 1e-3) / 1e12, "peak": tpeak, "unit": "TFLOP/s",
              "frac": flop_alg / (ct["ms_avg"] * 1e-3) / 1e12 / tpeak, "ms_per_launch": ct["ms_avg"],
              "note": "reference-defined dense FLOPs / time; ms_per_launch includes the plan + token pre-kernel"}

    variants = {}
    if not args.no_variants:
        # ---- the materialised layouts of the fine tracker's patch features, same values, same run ----
        for other in [l for l in ("up2", "cl", "nchw") if l != layout]:
            if other == "up2":
                continue   # (the headline was run with a materialised layout: the source map is not available)
            alt = upsample_fine(torch, devin["fine"]["fmaps"], other) if layout == "up2" else (
                devin["fine"]["fmaps"].contiguous() if other == "nchw"
                else devin["fine"]["fmaps"].permute(0, 1, 3, 4, 2).contiguous().permute(0, 1, 4, 2, 3))
            alt_in = {"coarse": devin["coarse"], "fine": dict(devin["fine"], fmaps=alt)}
            ms_alt, per_alt = timed(lambda: hp.run(alt_in), args.steps, args.warmup, per_class=True)
            variants["fine_" + other] = {
                "value": Q * world / (ms_alt * 1e-3), "unit": UNIT, "ms_per_step": ms_alt,
                "ms_per_step_by_class": {k: sum(v) / args.steps for k, v in per_alt.items()},
                "what": "same step with the fine tracker handed MATERIALISED 31x31 patch features, " +
                        ("NCHW-contiguous (the reference encoder's own output layout)" if other == "nchw"
                         else "as a channels-last view (a torch.channels_last encoder's output, zero-copy)")}
            del alt, alt_in
        # the reference's shipped configuration runs under torch.autocast(bf16) (mixed_precision: bf16, abl_ours.yaml:102):
        # CorrBlock.corr then rounds operands and volume to bf16.  Same step with that rounding mode selected.
        with torch.autocast("cuda", dtype=torch.bfloat16):
            ms_bf, per_bf = timed(step_dev, args.steps, args.warmup, per_class=True)
        variants["autocast_bf16"] = {"value": Q * world / (ms_bf * 1e-3), "unit": UNIT, "ms_per_step": ms_bf,
                                     "ms_per_step_by_class": {k: sum(v) / args.steps for k, v in per_bf.items()},
                                     "what": "same step under torch.autocast(bf16): one tensor-core pass, bf16-rounded "
                                             "operands and volume, fp32 lookup (parity bar 2e-2)"}

        # ---- B=1 (the reference's eval is hard-wired to batch 1): one sequence per step, eager and as ONE CUDA graph
        # replay of its launches (launch.CudaGraphRunner) ----
        one = {}
        for k, v in devin.items():
            nb = 1 if k == "coarse" else FINE["P"]
            one[k] = {"fmaps": v["fmaps"][:nb], "coords": v["coords"][:, :nb].contiguous(),
                      "feats": v["feats"][:, :nb].contiguous()}
        hp1 = HotPath(cb, torch, 1, dev)
        l0 = cb._lib.lib.comet_launch_count()
        hp1.run(one)
        n_launch1 = cb._lib.lib.comet_launch_count() - l0
        ms_b1, _ = timed(lambda: hp1.run(one), max(args.steps, 20), args.warmup)
        runner = cl.CudaGraphRunner(lambda: hp1.run(one))
        ms_g1, _ = timed(lambda: runner(), max(args.steps, 20), args.warmup)
        variants["batch1"] = {"value": world / (ms_b1 * 1e-3), "unit": UNIT, "ms_per_sequence": ms_b1,
                              "launches_per_sequence": int(n_launch1), "what": "one sequence per step, eager launches"}
        variants["batch1_graph"] = {"value": world / (ms_g1 * 1e-3), "unit": UNIT, "ms_per_sequence": ms_g1,
                                    "launches_per_sequence": int(n_launch1),
                                    "what": "one sequence per step, its launches captured once into a CUDA graph "
                                            "(launch.CudaGraphRunner) and replayed"}
        del runner, hp1, one

        # ---- config 4 (BASELINE.json configs[3]): long sequence, dense query grid -- S=64, N=4096 (64x64 grid at pixel
        # centres), coarse tracker only (the part that scales with S*N); per-iteration time and rates ----
        S4, N4 = 64, 4096
        g4 = torch.Generator(device=dev).manual_seed(4)
        fm4 = torch.randn(1, S4, COARSE["C"], 64, 64, device=dev, generator=g4)
        ys, xs = torch.meshgrid(torch.arange(64, device=dev), torch.arange(64, device=dev), indexing="ij")
        q4 = torch.stack([xs, ys], -1).reshape(1, 1, N4, 2).float() + 0.5          # pixel centres (8i+4, 8j+4) / 8
        co4 = (q4 + torch.randn(1, S4, N4, 2, device=dev, generator=g4) * 0.75)
        co4[:, 0] = q4[:, 0]
        ft4 = torch.randn(1, S4, N4, COARSE["C"], device=dev, generator=g4)
        out4 = torch.empty(1, N4, S4, hp.td_c, device=dev)
        blk4 = cb.CorrBlock(fm4, num_levels=COARSE["L"], radius=COARSE["r"])
        tk4 = cb.TrackTokenizer(blk4, co4[:, 0], hp.td_c)
        ms_c4, _ = timed(lambda: tk4.tokens(co4, ft4, out=out4), args.steps, args.warmup)
        flop4 = 2.0 * S4 * N4 * COARSE["C"] * 5456
        bytes4 = S4 * COARSE["C"] * 4096 * 4 + S4 * N4 * COARSE["C"] * 4 + S4 * N4 * 8 + N4 * S4 * hp.td_c * 4
        variants["config4"] = {"ms_per_iteration": ms_c4, "dense_equiv_TFLOPs": flop4 / (ms_c4 * 1e-3) / 1e12,
                               "frac_tensor_sustained": flop4 / (ms_c4 * 1e-3) / 1e12 / tpeak,
                               "compulsory_GBps": bytes4 / (ms_c4 * 1e-3) / 1e9, "frac_hbm": bytes4 / (ms_c4 * 1e-3) / 1e9 / peak,
                               "what": "coarse tracker, ONE sequence of S=64 frames with a dense 64x64 query grid (N=4096): "
                                       "one fused iteration (plan + tcgen05 corr + lookup + tokens); the reference "
                                       "materialises a 5.72 GB volume per iteration here"}
        del fm4, co4, ft4, out4, blk4, tk4

    # ---- the tracker loops WITH the update transformer (SURVEY 8f rank 1; outside `value`): drop-in BaseTrackerPredictor,
    # coarse (hidden 384, depth 6, 4 it, N=512) + fine (hidden 256, depth 4, 6 it, 512 patches on the 16x16 source map) of
    # ONE sequence, random-init weights; this package's sm_100a transformer kernels vs the torch.nn (cuBLAS / ATen)
    # definition of the same module, in float32 and under autocast(bf16) ----
    if not args.no_variants:
        from types import SimpleNamespace as NS
        import importlib

        ufm = importlib.import_module("comet_pose_estimation_b200.update_former")
        tcfg = NS(track_conf=False, MODEL=NS(TRACK=NS(efficient_corr=False)))
        torch.manual_seed(0)
        coarse_m = cb.BaseTrackerPredictor(cfg=tcfg, **TRACKER["coarse"]).eval().to(dev)
        fine_m = cb.BaseTrackerPredictor(cfg=tcfg, **TRACKER["fine"]).eval().to(dev)
        for mm in (coarse_m, fine_m):                      # small updates, as a trained tracker makes
            for prm in mm.updateformer.flow_head.parameters():
                prm.data.mul_(0.05)
        fm_c = devin["coarse"]["fmaps"][:1]
        qp_c = devin["coarse"]["coords"][0][:1, 0] * 8.0                      # pixels (stride 4 x down_ratio 2)
        src_f = devin["fine"]["fmaps"][:FINE["P"]]
        up_f = cb.Upsampled2x(src_f) if layout == "up2" else src_f
        qp_f = devin["fine"]["coords"][0][:FINE["P"], 0]

        def tracker_loops():
            with torch.no_grad():
                coarse_m(query_points=qp_c, fmaps=fm_c, iters=COARSE["iters"], down_ratio=2, TRACKorPOSE=False)
                fine_m(query_points=qp_f, fmaps=up_f, iters=FINE["iters"], TRACKorPOSE=False)

        tl = {}
        for tag, native, bf in (("sm100_kernels_fp32", True, False), ("torch_nn_fp32", False, False),
                                ("sm100_kernels_autocast_bf16", True, True), ("torch_nn_autocast_bf16", False, True)):
            ufm.USE_TC_KERNELS = native
            if bf:
                with torch.autocast("cuda", dtype=torch.bfloat16):
                    tl[tag], _ = timed(tracker_loops, 5, 2)
            else:
                tl[tag], _ = timed(tracker_loops, 5, 2)
        ufm.USE_TC_KERNELS = True
        variants["tracker_loop"] = {"ms_per_sequence": tl,
                                    "what": "coarse 4 it + fine 6 it of one 16-frame sequence through the drop-in "
                                            "BaseTrackerPredictor INCLUDING the update transformer and state updates: "
                                            "transformer on this package's tcgen05 / attention / LayerNorm kernels vs its "
                                            "torch.nn definition (cuBLAS / ATen); TF32 off for the float32 arms"}
        # ---- the whole tracker from IMAGES (process_images_to_fmaps -> coarse -> refine_track -> inverted score: the
        # tracker part of COMET.forward_all, E2Epose2.py:176-239) through TrackerPredictor.track, one 16-frame 512x512
        # sequence, device-resident and end to end from pinned host images (50 MB H2D, tracks + confidence D2H) ----
        tp = cb.TrackerPredictor(coarse_predictor=coarse_m, fine_predictor=fine_m, cfg=tcfg).eval().to(dev)
        tp.fine_fnet.to(memory_format=torch.channels_last)
        img_h = torch.rand(1, COARSE["S"], 3, 512, 512).pin_memory()
        q_h = (torch.rand(1, COARSE["N"], 2) * 480 + 16).pin_memory()
        img_d, q_d = img_h.to(dev), q_h.to(dev)
        res_h = torch.empty(1, COARSE["S"], COARSE["N"], 3).pin_memory()

        def from_images_dev():
            return tp.track(img_d, q_d, coarse_iters=COARSE["iters"])

        def from_images_host():
            o = tp.track(img_h.to(dev, non_blocking=True), q_h.to(dev, non_blocking=True), coarse_iters=COARSE["iters"])
            res_h[..., :2].copy_(o["refine_pred_track"], non_blocking=True)
            res_h[..., 2].copy_(o["pred_score"], non_blocking=True)

        fi = {}
        fi["ms_per_sequence"], _ = timed(from_images_dev, 5, 2)
        fi["ms_per_sequence_e2e_host_images"], _ = timed(from_images_host, 5, 2)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            fi["ms_per_sequence_autocast_bf16"], _ = timed(from_images_dev, 5, 2)
        fi["sequences_per_s"] = world / (fi["ms_per_sequence"] * 1e-3)
        fi["h2d_bytes"] = img_h.numel() * 4 + q_h.numel() * 4
        fi["d2h_bytes"] = res_h.numel() * 4
        fi["what"] = ("TrackerPredictor.track on one sequence of 16 512x512 frames, 512 query points: BasicEncoder (cuDNN convs, "
                      "library resize / instance-norm kernels) -> coarse tracker 4 it -> patch encoder -> fine tracker 6 it -> "
                      "score; random-init weights")
        variants["tracker_from_images"] = fi
        del coarse_m, fine_m, tp, img_d

    # ---- the producer of the fine tracker's input (SURVEY 8f rank 2, outside `value`): patch gather + ShallowEncoder for
    # ONE sequence (8192 patches of a 16-frame 512x512 sequence), with the library's resize / instance-norm kernels and
    # with the ATen ops the reference calls (F.interpolate, InstanceNorm2d) ----------------------------------------
    if not args.no_variants:
        import importlib

        rt = importlib.import_module("comet_pose_estimation_b200.refine_track")  # (the package exports a function of that name)
        torch.manual_seed(0)
        enc = rt.ShallowEncoder(3).eval().to(dev).to(memory_format=torch.channels_last)
        imgs = torch.rand(1, FINE["S"], 3, 512, 512, device=dev)
        tl = (torch.rand(1, FINE["S"], FINE["P"], 2, device=dev) * (512 - 31)).int()

        def producer(defer):
            with torch.no_grad():
                return enc(rt.extract_patches(imgs, tl, 31), defer_upsample=defer)

        def fused_from_images():
            with torch.no_grad():
                return enc.encode_patches_of(imgs, tl, defer_upsample=True)

        res = {}
        res["fused"], _ = timed(fused_from_images, 5, 10)
        res["fused_full_res"], _ = timed(lambda: producer(False), 5, 5)
        rt.USE_FUSED_ENCODER = False
        tf32 = torch.backends.cudnn.allow_tf32
        for tag, flag, defer, t32 in (("per_op_half_res_fp32", True, True, False), ("per_op_half_res_tf32", True, True, True),
                                      ("aten_ops", False, False, True)):
            rt.USE_LIBRARY_KERNELS = flag
            torch.backends.cudnn.allow_tf32 = t32
            res[tag], _ = timed(lambda: producer(defer), 3, 2)
        rt.USE_LIBRARY_KERNELS = True
        rt.USE_FUSED_ENCODER = True
        torch.backends.cudnn.allow_tf32 = tf32
        macs = FINE["S"] * FINE["P"] * 2.0398e6     # multiply-adds of the encoder's convolutions per sequence (DESIGN 5.4)
        variants["patch_encoder"] = {"ms_per_sequence_half_res_output": res["fused"],
                                     "ms_per_sequence": res["fused_full_res"],
                                     "fp32_fma_frac_of_peak": macs / (res["fused"] * 1e-3) / (148 * 128 * 1.965e9),
                                     "ms_per_sequence_per_operator_cudnn_fp32": res["per_op_half_res_fp32"],
                                     "ms_per_sequence_per_operator_cudnn_tf32": res["per_op_half_res_tf32"],
                                     "ms_per_sequence_aten_ops": res["aten_ops"],
                                     "what": "refine_track's producer of the fine tracker's input for one sequence (8192 "
                                             "patches of 31x31): the one-kernel float32 encoder (csrc/shallow_encoder.cu, "
                                             "patch gather fused) up to the 16x16 map the up2 layout consumes / "
                                             "extract_patches + encoder + the final 31x31 up-sampling / the per-operator "
                                             "path it replaced (gather kernel + cuDNN convolutions in strict float32 and "
                                             "in TF32 + the library's norm / resize kernels) / the ATen resize + "
                                             "instance-norm ops the reference calls"}
        del enc, imgs, tl

    # ---- end-to-end arm: host buffers, H2D + D2H inside the timed region ------------------------
    e2e = None
    if not args.no_e2e:
        def e2e_arm(host_in):
            out_c = torch.empty(hp.tok_c.shape, dtype=torch.float32).pin_memory()
            out_f = torch.empty(hp.tok_f.shape, dtype=torch.float32).pin_memory()
            h2d = sum(t.numel() * 4 for v in host_in.values() for t in v.values())
            d2h = out_c.numel() * 4 + out_f.numel() * 4
            # Two device-side staging sets: the H2D copy of step i+1 (copy stream) overlaps the kernels and the D2H of
            # step i (current stream).  Every step still copies all of its inputs from pinned host memory and reads its
            # result back; the pipeline fill (first copy) is inside the timed region.
            stages = [{k: {n: torch.empty_like(t, device=dev) for n, t in v.items()} for k, v in host_in.items()}
                      for _ in range(2)]
            copy_stream = torch.cuda.Stream(device=dev)
            copied = [torch.cuda.Event() for _ in range(2)]
            consumed = [torch.cuda.Event() for _ in range(2)]

            def issue_copy(i):
                with torch.cuda.stream(copy_stream):
                    copy_stream.wait_event(consumed[i % 2])       # the kernels of step i-2 are done with this set
                    for k, v in host_in.items():
                        for n, t in v.items():
                            stages[i % 2][k][n].copy_(t, non_blocking=True)
                    copied[i % 2].record(copy_stream)

            def e2e_run(nsteps):
                cur = torch.cuda.current_stream(dev)
                for ev in consumed:
                    ev.record(cur)
                issue_copy(0)
                for i in range(nsteps):
                    if i + 1 < nsteps:
                        issue_copy(i + 1)
                    cur.wait_event(copied[i % 2])
                    a, b = hp.run(stages[i % 2])
                    consumed[i % 2].record(cur)
                    out_c.copy_(a, non_blocking=True)
                    out_f.copy_(b, non_blocking=True)

            n_e2e = max(2, min(args.steps, 10))
            e2e_run(2)
            barrier()
            e0.record()
            e2e_run(n_e2e)
            e1.record()
            barrier()
            ms = max_over_ranks(e0.elapsed_time(e1)) / n_e2e
            return {"value": Q * world / (ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": ms, "steps": n_e2e,
                    "h2d_GBps_per_gpu": h2d / (ms * 1e-3) / 1e9}

        e2e = e2e_arm(host)
        e2e["api"] = ("CorrBlock%s + TrackTokenizer (ctypes -> C ABI), pinned host tensors; H2D of step i+1 overlapped "
                      "with the kernels / D2H of step i (two staging sets)" % (".from_upsampled" if layout == "up2" else ""))
        e2e["fine_layout"] = layout
        if layout == "up2" and not args.no_variants:
            # round-1 definition, kept for continuity: the MATERIALISED channels-last 31x31 patch features cross PCIe
            host_cl = dict(host, fine=dict(host["fine"]))
            up = upsample_fine(torch, host["fine"]["fmaps"], "cl")
            host_cl["fine"]["fmaps"] = torch.empty(up.permute(0, 1, 3, 4, 2).shape, dtype=torch.float32).pin_memory().permute(0, 1, 4, 2, 3)
            host_cl["fine"]["fmaps"].copy_(up)
            del up
            e2e["variants"] = {"fine_cl": e2e_arm(host_cl)}
            e2e["variants"]["fine_cl"]["what"] = ("round-1 definition: the materialised 31x31 channels-last patch features "
                                                   "(4x the bytes) are copied from the host every step")
            del host_cl

    if prev_affinity is not None:
        os.sched_setaffinity(0, prev_affinity)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, mean_s, ncores = cpu_reference_seq_per_s(torch, args.cpu_reps)
        cpu = {"value": v, "unit": UNIT, "cores": ncores, "kind": "port",
               "sample": f"1 sequence x {args.cpu_reps} reps (best), oracle/torch_port.py (reference's ATen calls), "
                         f"fp32, {mean_s:.2f} s/sequence mean"}
        if not args.no_variants:
            # BASELINE.md section 4 scope (ii): the tracker loops with the update transformer, one sequence, one rep
            cpu["tracker_loop_s_per_sequence"] = cpu_tracker_loop_s(torch, reps=1)
            cpu["tracker_loop_sample"] = ("scope (ii): coarse 4 it + fine 6 it of one sequence incl. the update transformer "
                                          "(torch.nn on the host cores) and state updates, best of 1 after a warm-up")
            # scope (iii): from images -- scope (ii) plus the two encoders on the host cores
            t_basic, t_shallow = cpu_encoders_s(torch)
            cpu["from_images_s_per_sequence"] = cpu["tracker_loop_s_per_sequence"] + t_basic + t_shallow
            cpu["from_images_sample"] = (f"scope (iii): scope (ii) + BasicEncoder on 16 frames of 512x512 ({t_basic:.2f} s) + ShallowEncoder "
                                         f"on 8192 patches of 31x31 ({t_shallow:.2f} s), torch.nn on the host cores, one pass each; "
                                         "compare variants.tracker_from_images")

    if rank == 0:
        config = make_config(Q, world, layout)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config,
            "fine_layout": layout + {"up2": " (the fine tracker reads the patch encoder's 16x16 output; levels 0/1 of the "
                                            "31x31 pyramid are evaluated inside the lookup, as comet_pose_estimation_b200."
                                            "refine_track does)",
                                     "cl": " (materialised 31x31 features, channels-last view)",
                                     "nchw": " (materialised 31x31 features, contiguous)"}[layout],
            "numa_bound": prev_affinity is not None,
            "roofline": roof, "rooflines": rooflines, "roofline_tensor": tensor, "variants": variants,
            "cpu_baseline": cpu, "e2e": e2e, "clocks": clocks,
            "gpu_launches": int(launches), "kernels": kern,
            "tensor_path": bool(cb._lib.lib.comet_has_tensor_path()),
        }
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
