"""Full-size (shipped-configuration) golden fixtures, produced by EXECUTING THE UNMODIFIED REFERENCE in float32 AND
in float64, plus the final-pose check-point.

Run in the build container only (needs /root/reference):

    python tests/golden/make_golden_full.py            # tracker_full.npz, refine_full.npz, pose.npz
    python tests/golden/make_golden_full.py --pose-from gpurun_out/cuda_tracks_full.npz   # adds the CUDA arm to pose.npz

What is stored (weights are NOT stored: ``cases.seeded_state_dict`` rebuilds them by parameter name on both sides):

* ``tracker_full.npz``  coarse ``BaseTrackerPredictor`` at hidden 384 / depth 6 / S=16 / N=512 / 4 iterations
  (abl_ours.yaml:99,399-428): per-iteration predicted tracks of the reference in float32 (``pred32_i``) and in
  float64 (``pred64_i``), visibility, a slice of the track features.  The float64 run is the yard-stick that turns
  the "any two fp32 implementations drift" statement of DESIGN.md section 3 into a measured bar:
  a conforming fp32 implementation must satisfy |impl - ref64| <= 3 |ref32 - ref64| per iteration.
  The query features and the track-feature slice are stored in ``tracker_full_feats.npz``.
* ``refine_full.npz``   ``refine_track`` (31x31 patches of 512x512 images -> ShallowEncoder -> fine tracker hidden 256 /
  depth 4 / 6 iterations (abl_ours.yaml:419-428) -> compute_score_fn) fed with the reference's own float32 coarse prediction: refined tracks
  and score in float32 and float64, and the inverted score of E2Epose2.py:232-236.
* ``pose.npz``          the wiring of ``COMET.forward_all`` after the tracker (E2Epose2.py:230-257) restated around
  the reference ``CameraPredictor`` (camera_predictor10.py:288-484) with a random-init stand-in for the DINOv2 backbone
  (SURVEY.md 8c; the backbone is shared by every arm, so it cancels): ``pred_pose_enc`` and ``pred_cameras.{R,T}`` for
  (a) the reference float32 tracks / score, (b) the reference float64 tracks / score (how far the pose moves under
  the reference's own fp32 rounding), (c) tracks / score produced by this repository's CUDA path on a B200 (copied
  back from the GPU box as ``cuda_tracks_full.npz``; the test that produced them is
  tests/test_full_size.py::test_full_chain_writes_tracks_for_pose_golden).
"""
from __future__ import annotations

import argparse
import os
import sys
import time
import types
from types import SimpleNamespace as NS

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import cases  # noqa: E402
import make_golden as mg  # noqa: E402  (import_reference, digest, save)

REF = mg.REF


def tracker_cfg():
    return NS(track_conf=False, MODEL=NS(TRACK=NS(efficient_corr=False)))


def load_seeded(module, seed, torch, gain=1.0):
    sd = cases.seeded_state_dict({k: tuple(v.shape) for k, v in module.state_dict().items()}, seed, gain)
    module.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()}, strict=True)
    return module


def install_kornia_stubs(torch):
    """kornia is not installed: the two functions refine_track.py:20-21 imports, restated from their documented
    semantics (SURVEY.md 8c) exactly as in make_golden.py."""

    def create_meshgrid(h, w, normalized_coordinates=True, device=None, dtype=torch.float32):
        xs = torch.linspace(-1, 1, w, device=device, dtype=dtype) if normalized_coordinates else torch.arange(w, device=device, dtype=dtype)
        ys = torch.linspace(-1, 1, h, device=device, dtype=dtype) if normalized_coordinates else torch.arange(h, device=device, dtype=dtype)
        gy, gx = torch.meshgrid(ys, xs, indexing="ij")
        return torch.stack([gx, gy], -1)[None]

    def spatial_expectation2d(heat, normalized_coordinates=True):
        b, n, h, w = heat.shape
        g = create_meshgrid(h, w, normalized_coordinates, heat.device, heat.dtype).reshape(-1, 2)
        flat = heat.reshape(b, n, -1)
        return torch.stack([(flat * g[:, 0]).sum(-1), (flat * g[:, 1]).sum(-1)], -1)

    for name in ("kornia", "kornia.utils", "kornia.utils.grid", "kornia.geometry", "kornia.geometry.subpix",
                 "kornia.geometry.subpix.dsnt"):
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.modules["kornia.utils.grid"].create_meshgrid = create_meshgrid
    sys.modules["kornia.geometry.subpix.dsnt"].spatial_expectation2d = spatial_expectation2d
    sys.modules["kornia.geometry.subpix"].dsnt = sys.modules["kornia.geometry.subpix.dsnt"]


class _F64Tables:
    """The reference builds its sin/cos tables in float64 and casts them to float32 (utils.py:724-755); F.grid_sample
    then refuses a float32 table with float64 coordinates.  For the float64 run the table is widened back (same
    values as the float32 run uses) -- the only change made to run the reference modules in double precision."""

    def __init__(self, module):
        self.module = module

    def __enter__(self):
        self.orig = self.module.get_2d_sincos_pos_embed
        self.module.get_2d_sincos_pos_embed = lambda *a, **k: self.orig(*a, **k).double()

    def __exit__(self, *exc):
        self.module.get_2d_sincos_pos_embed = self.orig


def run_coarse(torch, btp):
    t = torch.from_numpy
    m = load_seeded(btp.BaseTrackerPredictor(cfg=tracker_cfg(), **cases.FULL_COARSE_CTOR).eval(),
                    cases.FULL_SEEDS["coarse"], torch)
    fmaps, q = cases.tracker_case(**cases.FULL_COARSE_CASE)
    kw = dict(iters=cases.FULL_COARSE_ITERS, return_feat=True, down_ratio=cases.FULL_COARSE_CASE["down_ratio"],
              TRACKorPOSE=False)
    t0 = time.time()
    p32, vis32, tf32, qf32, _ = m(query_points=t(q), fmaps=t(fmaps), **kw)
    t1 = time.time()
    m = m.double()
    with _F64Tables(btp):
        p64, vis64, tf64, qf64, _ = m(query_points=t(q).double(), fmaps=t(fmaps).double(), **kw)
    print(f"coarse full: fp32 {t1 - t0:.1f} s, fp64 {time.time() - t1:.1f} s")
    out = {"digest": np.frombuffer(mg.digest(fmaps, q).encode(), dtype=np.uint8)}
    for i, (a, b) in enumerate(zip(p32, p64)):
        out[f"pred32_{i}"] = a.numpy()
        out[f"pred64_{i}"] = b.numpy()
        d = (a.double() - b).abs().max() / b.abs().max()
        print(f"  iteration {i}: |ref32 - ref64| / max|ref64| = {float(d):.3e}")
    out["vis32"], out["vis64"] = vis32.numpy(), vis64.numpy()
    mg.save("tracker_full", **out)
    # the features go to a file of their own: together with the tracks they exceed 1 MB
    mg.save("tracker_full_feats", digest=out["digest"], query_feat32=qf32.numpy(),
            track_feats32_slice=tf32[:, :, ::37].numpy(), track_feats64_slice=tf64[:, :, ::37].numpy())
    return p32[-1].numpy(), p64[-1].numpy()


def run_refine(torch, blocks, btp, coarse_pred, coarse_pred64):
    t = torch.from_numpy
    install_kornia_stubs(torch)
    import refine_track as rrt

    fnet = load_seeded(blocks.ShallowEncoder(input_dim=3).eval(), cases.FULL_SEEDS["fnet"], torch)
    ftr = load_seeded(btp.BaseTrackerPredictor(cfg=tracker_cfg(), **cases.FULL_FINE_CTOR).eval(),
                      cases.FULL_SEEDS["fine"], torch)
    images, _ = cases.refine_case(**cases.FULL_REFINE_CASE)
    coarse = np.clip(coarse_pred, 0.0, cases.FULL_REFINE_CASE["HW"] - 1.001).astype(np.float32)
    t0 = time.time()
    r32, s32 = rrt.refine_track(t(images), fnet, ftr, t(coarse), compute_score=True)
    t1 = time.time()
    fnet, ftr = fnet.double(), ftr.double()
    with _F64Tables(btp):
        r64, s64 = rrt.refine_track(t(images).double(), fnet, ftr, t(coarse).double(), compute_score=True)
        # the reference's own float64 CHAIN (float64 coarse prediction -> float64 refine_track): the yard-stick for an
        # implementation's chained output, whose coarse prediction differs from the float32 reference's by its drift
        c64 = np.clip(coarse_pred64, 0.0, cases.FULL_REFINE_CASE["HW"] - 1.001)
        r64c, s64c = rrt.refine_track(t(images).double(), fnet, ftr, t(c64), compute_score=True)
    print(f"refine full: fp32 {t1 - t0:.1f} s, fp64 (two runs) {time.time() - t1:.1f} s")

    def inverted(score):  # E2Epose2.py:232-236
        inv = 1.0 / (score + 1e-6)
        return inv / inv.max(dim=1, keepdim=True)[0]

    out = {"digest": np.frombuffer(mg.digest(images, coarse).encode(), dtype=np.uint8), "coarse_pred": coarse,
           "refined32": r32.numpy(), "refined64": r64.numpy(), "score32": s32.numpy(), "score64": s64.numpy(),
           "inverted32": inverted(s32).numpy(), "inverted64": inverted(s64).numpy(),
           "refined64_chain": r64c.numpy(), "score64_chain": s64c.numpy(), "inverted64_chain": inverted(s64c).numpy()}
    for k in ("refined", "score", "inverted"):
        a, b = out[k + "32"].astype(np.float64), out[k + "64"]
        print(f"  {k}: |ref32 - ref64| / max|ref64| = {np.abs(a - b).max() / np.abs(b).max():.3e}")
    mg.save("refine_full", **out)
    return images


class _Cfg(dict):
    """Minimal stand-in for the OmegaConf node CameraPredictor reads (``cfg.get(...)``, ``cfg.train.dataset``)."""

    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError as e:
            raise AttributeError(k) from e


def build_camera(torch):
    """Reference CameraPredictor (camera_predictor10.py:90-286) with a random-init stand-in backbone
    (SURVEY.md 8c: DINOv2 comes from torch.hub over the network; every arm shares this instance)."""
    import torch.nn as nn

    hydra = types.ModuleType("hydra")
    hydra.utils = types.ModuleType("hydra.utils")
    hydra.utils.instantiate = lambda *a, **k: None
    sys.modules.setdefault("hydra", hydra)
    sys.modules.setdefault("hydra.utils", hydra.utils)

    class QuaternionCameras:  # the container pose_encoding_to_camera2 fills (train_eval_func.py:113-160)
        def __init__(self, R=None, T=None, focal_length=None, device=None, **kw):
            self.R, self.T, self.focal_length = R, T, focal_length

    sys.modules["train_eval_func"].QuaternionCameras = QuaternionCameras
    from models import camera_predictor10 as cp

    # the reference file is importable under several module names (SURVEY.md 3.3); patch the one the predictor uses
    cp.pose_encoding_to_camera2.__globals__["QuaternionCameras"] = QuaternionCameras

    class Backbone(nn.Module):  # 14x14 patchify of the 336x336 input -> (BS, 576, 768) "x_norm_patchtokens"
        def __init__(self):
            super().__init__()
            self.proj = nn.Conv2d(3, 768, kernel_size=14, stride=14)
            self.norm = nn.LayerNorm(768)

        def forward(self, x, is_training=True):
            return {"x_norm_patchtokens": self.norm(self.proj(x).flatten(2).transpose(1, 2))}

    cp.CameraPredictor.get_backbone = lambda self, name: Backbone()
    cfg = _Cfg(train=_Cfg(dataset="AMD_eval"))
    cam = cp.CameraPredictor(cfg=cfg).eval()   # defaults = abl_ours.yaml:430-431
    return load_seeded(cam, cases.FULL_SEEDS["camera"], torch)


def gt_cameras_stub(torch, S):
    rng = np.random.default_rng(81)
    q = rng.standard_normal((S, 4))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    T = np.tile(np.array([[320.0, 240.0, 10.0]]), (S, 1))
    return NS(R=torch.from_numpy(q.astype(np.float32)), T_uvz=torch.from_numpy(T.astype(np.float32)), ratio=1.3)


def run_pose(torch, images, arms):
    """arms: {name: (tracks (1,S,N,2) float32, inverted score (1,S,N) float32)} -> pose per arm."""
    cam = build_camera(torch)
    B, S, C, H, W = images.shape
    gt = gt_cameras_stub(torch, S)
    from models import camera_predictor10 as cp

    # camera_to_pose_encoding2 needs the real camera classes only to produce gt_pose_enc for the loss; not the
    # check-point -> identity stand-in returning zeros of the right shape
    cp.camera_to_pose_encoding2 = lambda cams, pose_encoding_type=None: torch.zeros(S, 7)
    out = {}
    img = torch.from_numpy(images).reshape(-1, C, H, W)
    for name, (tracks, conf) in arms.items():
        t0 = time.time()
        res = cam(img, preliminary_cameras=None, batch_size=B, gt_cameras=gt, iters=4,
                  pred_trajectories=torch.from_numpy(tracks), track_confidence=torch.from_numpy(conf))
        out[name + "/pred_pose_enc"] = res["pred_pose_enc"].numpy()
        out[name + "/R"] = res["pred_cameras"].R.numpy()
        out[name + "/T"] = res["pred_cameras"].T.numpy()
        print(f"pose arm {name}: {time.time() - t0:.1f} s")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pose-from", default=None, help="npz with CUDA-produced 'refined' and 'inverted' (GPU box output)")
    ap.add_argument("--only-pose", action="store_true")
    args = ap.parse_args()
    import torch

    torch.manual_seed(0)
    torch.set_grad_enabled(False)
    blocks, btp, ru = mg.import_reference()
    if not args.only_pose:
        coarse_pred, coarse_pred64 = run_coarse(torch, btp)
        images = run_refine(torch, blocks, btp, coarse_pred, coarse_pred64)
    else:
        images, _ = cases.refine_case(**cases.FULL_REFINE_CASE)
    g = np.load(os.path.join(HERE, "refine_full.npz"))
    arms = {"ref32": (g["refined32"], g["inverted32"]),
            "ref64": (g["refined64"].astype(np.float32), g["inverted64"].astype(np.float32)),
            "ref64_chain": (g["refined64_chain"].astype(np.float32), g["inverted64_chain"].astype(np.float32))}
    if args.pose_from:
        c = np.load(args.pose_from)
        arms["cuda"] = (c["refined"].astype(np.float32), c["inverted"].astype(np.float32))
        arms["cuda_chain"] = (c["refined_chain"].astype(np.float32), c["inverted_chain"].astype(np.float32))
    out = run_pose(torch, images, arms)
    ref = out["ref32/pred_pose_enc"].astype(np.float64)
    for name in arms:
        if name == "ref32":
            continue
        for k in ("pred_pose_enc", "R", "T"):
            a, b = out[f"{name}/{k}"].astype(np.float64), out[f"ref32/{k}"].astype(np.float64)
            print(f"  pose {name} vs ref32, {k}: max|a-b|/max|b| = {np.abs(a - b).max() / np.abs(b).max():.3e}")
    mg.save("pose", **out)


if __name__ == "__main__":
    main()
