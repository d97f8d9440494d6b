"""Drop-in ``TrackerPredictor`` container and ``BasicEncoder`` (comet/models/track_predictor.py:16-151,
comet/models/track_modules/blocks.py:27-111) -- the step right before the hot path (SURVEY.md section 8f, rank 4) -- and
the tracker part of ``COMET.forward_all`` (comet/models/E2Epose2.py:176-239) as one call.

What is B200-specific: its four bilinear resizes to 1/stride resolution
(blocks.py:99-102, ``_bilinear_intepolate`` :198-201) and its instance norms run in this library's kernels
(``comet_upsample_bilinear_ac_f32``, ``comet_instance_norm_f32``: ATen's up-sampling kernel walks batch x channels inside
every thread); the convolutions stay cuDNN.  Parameter names are the reference's (``conv1``, ``layer{1..4}.{0,1}.conv{1,2}``,
``layer*.0.downsample.0``, ``conv2``, ``conv3``), so ``track_predictor.coarse_fnet.*`` checkpoints load unchanged.

The reference builds the four sub-modules with ``hydra.utils.instantiate`` from the ``COARSE`` / ``FINE`` config nodes
(track_predictor.py:48-62); here they are passed in (or built with the shipped defaults of abl_ours.yaml:399-428), so no
hydra dependency is needed.
"""
from __future__ import annotations

from types import SimpleNamespace

import torch
import torch.nn as nn
import torch.nn.functional as F

from .base_track_predictor import BaseTrackerPredictor
from .refine_track import ShallowEncoder, _inorm, _ResidualBlock, _resize, inverted_score, refine_track
from .utils import check_num_tracks, check_query_frames, query_frame_items


class BasicEncoder(nn.Module):
    """blocks.py:27-111 (``norm_fn="instance"``, the only value the reference uses)."""

    def __init__(self, input_dim=3, output_dim=128, stride=4, use_trans=False, cfg=None):
        super().__init__()
        self.stride = stride
        self.norm_fn = "instance"
        self.in_planes = output_dim // 2
        self.norm1 = nn.InstanceNorm2d(self.in_planes)
        self.norm2 = nn.InstanceNorm2d(output_dim * 2)
        self.conv1 = nn.Conv2d(input_dim, self.in_planes, kernel_size=7, stride=2, padding=3)
        self.layer1 = self._make_layer(output_dim // 2, stride=1)
        self.layer2 = self._make_layer(output_dim // 4 * 3, stride=2)
        self.layer3 = self._make_layer(output_dim, stride=2)
        self.layer4 = self._make_layer(output_dim, stride=2)
        self.conv2 = nn.Conv2d(output_dim * 3 + output_dim // 4, output_dim * 2, kernel_size=3, padding=1)
        self.conv3 = nn.Conv2d(output_dim * 2, output_dim, kernel_size=1)
        for m in self.modules():
            if isinstance(m, nn.Conv2d):
                nn.init.kaiming_normal_(m.weight, mode="fan_out", nonlinearity="relu")

    def _make_layer(self, dim, stride=1):
        layers = (_ResidualBlock(self.in_planes, dim, stride=stride), _ResidualBlock(dim, dim, stride=1))
        self.in_planes = dim
        return nn.Sequential(*layers)

    def forward(self, x):
        _, _, H, W = x.shape
        size = (H // self.stride, W // self.stride)
        x = _inorm(self.norm1, self.conv1(x), True)
        a = self.layer1(x)
        b = self.layer2(a)
        c = self.layer3(b)
        d = self.layer4(c)
        x = torch.cat([_resize(a, size), _resize(b, size), _resize(c, size), _resize(d, size)], dim=1)
        x = _inorm(self.norm2, self.conv2(x), True)
        return self.conv3(x)


def _default_cfg():
    return SimpleNamespace(track_conf=False, MODEL=SimpleNamespace(TRACK=SimpleNamespace(efficient_corr=False)))


class TrackerPredictor(nn.Module):
    """track_predictor.py:16-151.  Attribute names (``coarse_fnet``, ``coarse_predictor``, ``fine_fnet``,
    ``fine_predictor``, ``coarse_down_ratio``) are the reference's; sub-modules not passed in are built with the shipped
    configuration (abl_ours.yaml:399-428)."""

    def __init__(self, coarse_fnet=None, coarse_predictor=None, fine_fnet=None, fine_predictor=None, coarse_stride=4,
                 coarse_down_ratio=2, cfg=None):
        super().__init__()
        self.cfg = cfg if cfg is not None else _default_cfg()
        self.coarse_down_ratio = coarse_down_ratio
        self.coarse_fnet = coarse_fnet if coarse_fnet is not None else BasicEncoder(stride=coarse_stride, cfg=self.cfg)
        self.coarse_predictor = coarse_predictor if coarse_predictor is not None else BaseTrackerPredictor(
            stride=coarse_stride, cfg=self.cfg)
        self.fine_fnet = fine_fnet if fine_fnet is not None else ShallowEncoder(input_dim=3, stride=1, cfg=self.cfg)
        self.fine_predictor = fine_predictor if fine_predictor is not None else BaseTrackerPredictor(
            stride=1, depth=4, corr_levels=3, corr_radius=3, latent_dim=32, hidden_size=256, fine=True,
            use_spaceatt=False, cfg=self.cfg)

    def process_images_to_fmaps(self, images, training=False):
        """track_predictor.py:117-151: (B,S,3,H,W) -> (B,S,128,H/(stride*down_ratio),W/(stride*down_ratio))."""
        B, S, C, H, W = images.shape
        if not training:
            assert B == 1, "now we only support processing one scene during inference"
        return self._encode_frames(images)

    def _encode_frames(self, images, frames=None):
        """(B,S,3,H,W) -> (B,S,128,h,w): one encoder call over all B*S frames.  ``frames`` (B ints): only the first
        frames[b] frames of sequence b are read and encoded (in one call: the instance norms are per frame); the maps of
        the others are zeros."""
        B, S, C, H, W = images.shape
        if frames is not None:
            fm = self._encode_frames(torch.cat([images[b, :n] for b, n in enumerate(frames)])[None])[0]
            out = fm.new_zeros((B, S) + tuple(fm.shape[1:]))
            at = 0
            for b, n in enumerate(frames):
                out[b, :n] = fm[at:at + n]
                at += n
            return out
        x = images.reshape(B * S, C, H, W)
        if self.coarse_down_ratio > 1:
            # F.interpolate(scale_factor=1/down_ratio, bilinear, align_corners=True): output size floor(H / down_ratio)
            x = _resize(x, (int(H * (1.0 / self.coarse_down_ratio)), int(W * (1.0 / self.coarse_down_ratio))))
        # NCHW on purpose: the channels-last instance-norm kernel of this library is built for the patch encoder's many tiny
        # planes (one thread per (sample, channel)); at 16 x 64 planes of 256 x 256 it would take 20 ms (measured), the
        # NCHW kernel (one warp per plane) 2.9 ms for the whole encoder (torch ops: 5.5 ms)
        fmaps = self.coarse_fnet(x.contiguous())
        return fmaps.reshape(B, S, -1, fmaps.shape[-2], fmaps.shape[-1])

    @torch.no_grad()
    def track(self, images, query_points, coarse_iters=4, fine_tracking=True, query_frames=None):
        """The tracker part of ``COMET.forward_all`` (E2Epose2.py:176-239): images (B,S,3,H,W) in the model's
        normalisation, ``query_points`` (B,N,2) pixels of frame 0 -> dict with ``coarse_pred_track`` /
        ``refine_pred_track`` (B,S,N,2), ``pred_score`` (the inverted, normalised track confidence the camera predictor
        consumes), ``vis`` and the per-iteration coarse list.

        ``query_frames`` ((1, N) or (N,) integers): track n starts on frame ``query_frames[n]`` and ``query_points[:, n]``
        are pixels of that frame; see ``track_batch``.  The dict then also holds ``query_frames`` (1, N) int64."""
        if query_frames is not None:
            assert images.shape[0] == 1, "now we only support processing one scene during inference"
            qf = query_frames.reshape(1, -1) if isinstance(query_frames, torch.Tensor) else torch.tensor([list(query_frames)])
            return split_batch(self.track_batch(images, query_points, coarse_iters=coarse_iters, fine_tracking=fine_tracking,
                                                query_frames=qf))[0]
        fmaps = self.process_images_to_fmaps(images)
        coarse_list, vis, track_feats, query_feat, conf = self.coarse_predictor(
            query_points=query_points, fmaps=fmaps, iters=coarse_iters, down_ratio=self.coarse_down_ratio, is_train=False,
            return_feat=True, TRACKorPOSE=False)
        coarse = coarse_list[-1]
        out = {"coarse_pred_track_list": coarse_list, "coarse_pred_track": coarse, "vis": vis, "conf": conf}
        if fine_tracking:
            refined, score = refine_track(images, self.fine_fnet, self.fine_predictor, coarse, compute_score=True)
            out["refine_pred_track"] = refined
            out["track_score"] = score
            out["pred_score"] = inverted_score(score)
        else:
            out["refine_pred_track"] = coarse
            out["pred_score"] = torch.ones_like(vis)
        return out

    @torch.no_grad()
    def track_batch(self, images, query_points, num_tracks=None, coarse_iters=4, fine_tracking=True, num_frames=None,
                    query_frames=None):
        """``track`` for B sequences in one call: images (B,S,3,H,W) (same image size for all), ``query_points``
        a list of B tensors (N_b, 2) or a padded (B, N_max, 2) tensor with ``num_tracks`` (B,) (None: every sequence
        has N_max tracks).  Returns ``track``'s dict with padded tensors (entries of tracks n >= N_b are 0) plus
        ``num_tracks`` (B,) int64; ``split_batch`` cuts it into per-sequence dicts.  Sequence b gets what ``track``
        returns for it alone (up to the rounding of the iterated loop).

        Sequences of different lengths: ``images`` a list of B tensors (S_b,3,H,W), or the padded (B,S_max,3,H,W) with
        ``num_frames`` (B,) (1 <= S_b <= S_max).  Frames s >= S_b of a padded tensor are never read; every output entry
        of such a frame is 0, ``pred_score`` is normalised over the real frames of each track, and the dict gets
        ``num_frames`` (B,) int64.

        Tracks that start on any frame: ``query_frames`` gives each track's query frame t_n (a list of B integer tensors
        (N_b,), or a padded (B, N_max) tensor; None: all 0), and ``query_points`` are pixels of that frame.  Track n of
        sequence b with t_n = q gets what this call returns for it on one item: sequence b's images with frames 0 and q
        swapped, the tracks of sequence b whose query frame is q (in their order), S_b frames -- with every per-frame
        output swapped back.  Tracks of different query frames do not interact.  The frames are encoded once whatever
        the number of query frames; every item reads them through a frame table.  The dict gets ``query_frames``
        (B, N_max) int64.  Query frames all 0 run exactly the path without them."""
        if isinstance(images, (list, tuple)):
            slens = [int(x.shape[0]) for x in images]
            assert num_frames is None or check_num_tracks(num_frames, len(images), max(slens)) == slens, \
                "num_frames disagrees with the image lists"
            padded = images[0].new_zeros((len(images), max(slens)) + tuple(images[0].shape[1:]))
            for b, x in enumerate(images):
                padded[b, :x.shape[0]] = x
            images, num_frames = padded, slens
        B, S = images.shape[:2]
        frames = None if num_frames is None else check_num_tracks(num_frames, B, S)
        if isinstance(query_points, (list, tuple)):
            assert len(query_points) == B, f"{len(query_points)} query tensors for {B} sequences"
            lens = [int(q.shape[0]) for q in query_points]
            assert num_tracks is None or check_num_tracks(num_tracks, B, max(lens)) == lens, \
                "num_tracks disagrees with the query lists"
            padded = query_points[0].new_zeros((B, max(lens), 2))
            for b, q in enumerate(query_points):
                padded[b, :q.shape[0]] = q
            query_points = padded
            num_tracks = lens
        assert query_points.dim() == 3 and query_points.shape[0] == B and query_points.shape[2] == 2
        N = query_points.shape[1]
        counts = check_num_tracks([N] * B if num_tracks is None else num_tracks, B, N)
        if query_frames is not None:
            qf = check_query_frames(query_frames, counts, [S] * B if frames is None else frames)
            if any(t for q in qf for t in q):
                return self._track_batch_query_frames(images, query_points, counts, frames, qf, coarse_iters, fine_tracking)
            out = self.track_batch(images, query_points, counts, coarse_iters, fine_tracking, frames)
            out["query_frames"] = torch.zeros((B, N), dtype=torch.int64)
            return out
        if frames is not None:
            return self._track_batch_frames(images, query_points, counts, frames, coarse_iters, fine_tracking)
        fmaps = self._encode_frames(images)
        coarse_list, vis, track_feats, query_feat, conf = self.coarse_predictor(
            query_points=query_points, fmaps=fmaps, iters=coarse_iters, down_ratio=self.coarse_down_ratio, is_train=False,
            return_feat=True, TRACKorPOSE=False, num_tracks=counts)
        coarse = coarse_list[-1]
        out = {"coarse_pred_track_list": coarse_list, "coarse_pred_track": coarse, "vis": vis, "conf": conf}
        if fine_tracking:
            refined, score = refine_track(images, self.fine_fnet, self.fine_predictor, coarse, compute_score=True,
                                          num_tracks=counts)
            real = (torch.arange(N, device=coarse.device)[None, :] < torch.tensor(counts, device=coarse.device)[:, None])
            out["refine_pred_track"] = refined
            out["track_score"] = score
            out["pred_score"] = inverted_score(score) * real[:, None, :]
        else:
            out["refine_pred_track"] = coarse
            real = (torch.arange(N, device=coarse.device)[None, :] < torch.tensor(counts, device=coarse.device)[:, None])
            out["pred_score"] = torch.ones_like(vis) * real[:, None, :]
        out["num_tracks"] = torch.tensor(counts, dtype=torch.int64)
        return out

    def _track_batch_frames(self, images, query_points, counts, frames, coarse_iters, fine_tracking):
        """``track_batch`` with per-sequence frame counts (validated lists)."""
        B, S = images.shape[:2]
        N = query_points.shape[1]
        fmaps = self._encode_frames(images, frames)
        coarse_list, vis, track_feats, query_feat, conf = self.coarse_predictor(
            query_points=query_points, fmaps=fmaps, iters=coarse_iters, down_ratio=self.coarse_down_ratio, is_train=False,
            return_feat=True, TRACKorPOSE=False, num_tracks=counts, num_frames=frames)
        coarse = coarse_list[-1]
        out = {"coarse_pred_track_list": coarse_list, "coarse_pred_track": coarse, "vis": vis, "conf": conf}
        real = padded_mask(counts, frames, S, N, coarse.device)
        if fine_tracking:
            refined, score = refine_track(images, self.fine_fnet, self.fine_predictor, coarse, compute_score=True,
                                          num_tracks=counts, num_frames=frames)
            out["refine_pred_track"] = refined
            out["track_score"] = score
            out["pred_score"] = inverted_score_padded(score, real)
        else:
            out["refine_pred_track"] = coarse
            out["pred_score"] = torch.ones_like(vis) * real
        out["num_tracks"] = torch.tensor(counts, dtype=torch.int64)
        out["num_frames"] = torch.tensor(frames, dtype=torch.int64)
        return out


    def _track_batch_query_frames(self, images, query_points, counts, frames, qf, coarse_iters, fine_tracking):
        """``track_batch`` with per-track query frames (validated lists): one item per (sequence, query frame), one
        encoder pass over the source frames, one predictor and one ``refine_track`` call over the items, results
        scattered back to (sequence, frame, track) order."""
        B, S = images.shape[:2]
        N = query_points.shape[1]
        dev = query_points.device
        items, frame_index = query_frame_items(qf, [S] * B if frames is None else frames, S)
        item_counts = [len(ns) for _, _, ns in items]
        item_frames = None if frames is None else [frames[b] for b, _, _ in items]
        item_b = torch.tensor([b for b, _, ns in items for _ in ns], device=dev)        # (M,) per real track
        item_i = torch.tensor([i for i, (_, _, ns) in enumerate(items) for _ in ns], device=dev)
        item_j = torch.tensor([j for _, _, ns in items for j in range(len(ns))], device=dev)
        item_n = torch.tensor([n for _, _, ns in items for n in ns], device=dev)
        q_items = query_points.new_zeros((len(items), max(item_counts), 2))
        q_items[item_i, item_j] = query_points[item_b, item_n]
        # position s of item i shows frame swap(s) of its sequence, and the swap is its own inverse
        pos_of_frame = (frame_index - torch.tensor([b * S for b, _, _ in items])[:, None]).to(dev)   # (B', S)

        fmaps = self._encode_frames(images, frames)
        coarse_list, vis, track_feats, query_feat, conf = self.coarse_predictor(
            query_points=q_items, fmaps=fmaps, iters=coarse_iters, down_ratio=self.coarse_down_ratio, is_train=False,
            return_feat=True, TRACKorPOSE=False, num_tracks=item_counts, num_frames=item_frames, frame_index=frame_index)
        coarse = coarse_list[-1]
        Si, Ni = coarse.shape[1], coarse.shape[2]
        out = {"coarse_pred_track_list": coarse_list, "coarse_pred_track": coarse, "vis": vis, "conf": conf}
        real = padded_mask(item_counts, [Si] * len(items) if item_frames is None else item_frames, Si, Ni, coarse.device)
        if fine_tracking:
            refined, score = refine_track(images, self.fine_fnet, self.fine_predictor, coarse, compute_score=True,
                                          num_tracks=item_counts, num_frames=item_frames, frame_index=frame_index)
            out["refine_pred_track"] = refined
            out["track_score"] = score
            out["pred_score"] = inverted_score(score) * real if item_frames is None else inverted_score_padded(score, real)
        else:
            out["refine_pred_track"] = coarse
            out["pred_score"] = torch.ones_like(vis) * real

        def scatter(v):
            if v is None:
                return None
            if isinstance(v, list):
                return [scatter(x) for x in v]
            idx = pos_of_frame.reshape(pos_of_frame.shape + (1,) * (v.dim() - 2)).expand((-1, -1) + tuple(v.shape[2:]))
            v = v.gather(1, idx)                                    # (B', S, N_cap, ...) in each sequence's frame order
            res = v.new_zeros((B, S, N) + tuple(v.shape[3:]))
            res[item_b, :, item_n] = v[item_i, :, item_j]
            return res

        out = {k: scatter(v) for k, v in out.items()}
        out["num_tracks"] = torch.tensor(counts, dtype=torch.int64)
        if frames is not None:
            out["num_frames"] = torch.tensor(frames, dtype=torch.int64)
        qf_pad = torch.zeros((B, N), dtype=torch.int64)
        for b, q in enumerate(qf):
            qf_pad[b, :len(q)] = torch.tensor(q, dtype=torch.int64)
        out["query_frames"] = qf_pad
        return out


def padded_mask(counts, frames, S: int, N: int, device) -> torch.Tensor:
    """(B, S, N) bool: entry (b, s, n) is a real frame and track of a padded batch."""
    c = torch.tensor(counts, device=device)
    f = torch.tensor(frames, device=device)
    return ((torch.arange(S, device=device)[None, :, None] < f[:, None, None])
            & (torch.arange(N, device=device)[None, None, :] < c[:, None, None]))


def inverted_score_padded(track_score: torch.Tensor, real: torch.Tensor, eps: float = 1e-6) -> torch.Tensor:
    """``inverted_score`` of a padded batch: each track normalised by its maximum over its real frames only (a padded
    score of 0 would invert to 1e6 and become the maximum); padded entries are 0."""
    inv = (1.0 / (track_score + eps)).masked_fill(~real, 0.0)
    m = inv.max(dim=1, keepdim=True)[0]
    return inv / torch.where(m > 0, m, torch.ones_like(m))


def split_batch(out):
    """``track_batch``'s padded dict -> list of per-sequence dicts with exactly ``track``'s keys and shapes (cut along
    the frame axis too when the dict has ``num_frames``; ``query_frames`` is cut to (1, N_b))."""
    counts = [int(n) for n in out["num_tracks"]]
    frames = [int(s) for s in out["num_frames"]] if "num_frames" in out else [None] * len(counts)

    def cut(v, b, n, s):
        if v is None:
            return None
        if isinstance(v, list):
            return [cut(x, b, n, s) for x in v]
        if v.dim() == 2:                                    # per-track keys (B, N_max): query_frames
            return v[b:b + 1, :n]
        return v[b:b + 1, :s, :n]

    return [{k: cut(v, b, n, s) for k, v in out.items() if k not in ("num_tracks", "num_frames")}
            for b, (n, s) in enumerate(zip(counts, frames))]
