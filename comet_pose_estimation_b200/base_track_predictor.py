"""Drop-in ``BaseTrackerPredictor`` (comet/models/track_modules/base_track_predictor.py:15-284).

Same constructor, ``forward`` signature, return tuple and state-dict keys (``updateformer.*``, ``norm.*``,
``ffeat_updater.0.*``, ``vis_predictor.0.*``, ``conf_predictor.0.*``).  Per refinement iteration the reference
issues ~25 ATen kernels plus a host-built, re-uploaded 10.9 MB sin/cos table (SURVEY 3.1); here the hot path is:

    once per call    pyramid (+ hi/lo split for the tensor path), sampled position embedding, query features
    per iteration    ONE fused kernel -> tokens (B,N,S,D), then the update transformer and the state update

The loop-state arithmetic (coords += delta, track_feats += ffeat_updater(norm(delta_feat)), frame 0 pinned,
rescale to pixels, base_track_predictor.py:229-262) is kept operation for operation.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from .blocks import CorrBlock, EfficientCorrBlock, Upsampled2x
from .track_tokens import TrackTokenizer, transformer_dim
from .update_former import EfficientUpdateFormer
from .utils import sample_features4d


class BaseTrackerPredictor(nn.Module):
    def __init__(self, stride=4, corr_levels=5, corr_radius=4, latent_dim=128, hidden_size=384, use_spaceatt=True,
                 depth=6, fine=False, cfg=None, updateformer_cls=EfficientUpdateFormer):
        super().__init__()
        self.cfg = cfg
        self.stride = stride
        self.latent_dim = latent_dim
        self.corr_levels = corr_levels
        self.corr_radius = corr_radius
        self.hidden_size = hidden_size
        self.fine = fine
        self.flows_emb_dim = latent_dim // 2
        self.transformer_dim = transformer_dim(corr_levels, corr_radius, latent_dim, fine)
        self.efficient_corr = cfg.MODEL.TRACK.efficient_corr  # config key MODEL.TRACK.efficient_corr (abl_ours.yaml:401)
        space_depth = depth if use_spaceatt else 0
        self.updateformer = updateformer_cls(
            space_depth=space_depth, time_depth=depth, input_dim=self.transformer_dim, hidden_size=hidden_size,
            output_dim=latent_dim + 2, mlp_ratio=4.0, add_space_attn=use_spaceatt)
        self.norm = nn.GroupNorm(1, latent_dim)
        self.ffeat_updater = nn.Sequential(nn.Linear(latent_dim, latent_dim), nn.GELU())
        if self.cfg.track_conf:  # config key track_conf (abl_ours.yaml:380)
            self.conf_predictor = nn.Sequential(nn.Linear(latent_dim, 1))
        if not self.fine:
            self.vis_predictor = nn.Sequential(nn.Linear(latent_dim, 1))

    def forward(self, query_points, fmaps=None, iters=4, return_feat=False, down_ratio=1, is_train=False,
                track_feats=None, TRACKorPOSE=True, ind=0, num_tracks=None, num_frames=None, frame_index=None,
                group_items=None):
        """``num_tracks`` (B ints or a 1-D tensor, ``TRACKorPOSE=False`` only): ``query_points`` (B, N_max, 2) is a padded
        batch of sequences with different track counts.  Sequence b's tracks get what a call on that sequence alone
        computes (up to rounding); every output entry of a padded track (n >= num_tracks[b]) is 0.  ``num_frames``
        (likewise): sequence b has the first ``num_frames[b]`` of the S frames of ``fmaps``; every output entry of a padded
        frame is 0, and the tracks of padded frames start at 0 and receive zero updates.

        ``frame_index`` ((B', S) integer tensor, ``TRACKorPOSE=False`` only): ``fmaps`` (B_src, S_src, C, H, W) holds
        source frames (any S_src) and ``query_points`` (B', N_max, 2) a batch of B' items of S positions; item i sees
        source frame ``frame_index[i, s]`` (flat index into the B_src * S_src frames) at position s, and any source frame
        may appear any number of times.  The result is the forward on the gathered maps
        ``fmaps.flatten(0, 1)[frame_index]``: on the GPU the pyramid is prepared once over the source frames and the token
        kernels read it through the table; elsewhere the gathered maps are built and the ordinary path runs.

        Size groups (``TRACKorPOSE=False`` only): ``fmaps`` a list of G per-group maps (B_g, S, C, H_g, W_g) of different
        sizes, and the items of ``query_points`` ordered group by group -- B_g items per group, or ``group_items[g]``
        with ``frame_index``, whose rows of group g index group g's B_g * S_g source frames (S_g may differ per group).  Each item gets what the call on its
        group alone computes (up to the rounding of the iterated loop; tokens and the first transformer pass are the
        same bits): every group has its own pyramid, position embedding and token launch, and the update transformer
        runs once over all items.  Elsewhere than on the GPU each group runs alone and the results are concatenated."""
        if frame_index is not None and not isinstance(fmaps, (list, tuple)):
            fmaps, group_items = [fmaps], [query_points.shape[0]]         # one source pool: a single size group
        grouped = isinstance(fmaps, (list, tuple))
        if grouped:
            assert not TRACKorPOSE, "size groups and frame_index are served with TRACKorPOSE=False only"
            fmaps = list(fmaps)
            Bi = query_points.shape[0]
            sizes = [f.shape[0] for f in fmaps] if group_items is None else [int(n) for n in group_items]
            assert frame_index is None or group_items is not None, "frame_index over size groups needs group_items"
            assert len(sizes) == len(fmaps) and all(n >= 1 for n in sizes) and sum(sizes) == Bi, \
                f"group_items {sizes} do not cover the {Bi} items"
            assert frame_index is not None or all(f.shape[0] == n for f, n in zip(fmaps, sizes))
            assert all(f.dim() == 5 and (frame_index is not None or f.shape[1] == fmaps[0].shape[1]) for f in fmaps), \
                "per-group fmaps (B_g, S, C, H, W)"
            if frame_index is not None:
                assert frame_index.dim() == 2 and frame_index.shape[0] == Bi, \
                    f"frame_index must be (B', S) with B' = {Bi}, got {tuple(frame_index.shape)}"
            B_items, S_maps = Bi, fmaps[0].shape[1] if frame_index is None else frame_index.shape[1]
            if not fmaps[0].is_cuda:
                from .utils import check_num_tracks

                counts = None if num_tracks is None else check_num_tracks(num_tracks, Bi, query_points.shape[1])
                frames = None if num_frames is None else check_num_tracks(num_frames, Bi, S_maps)
                outs, at = [], 0
                for f, n in zip(fmaps, sizes):
                    if frame_index is not None:
                        f = f.flatten(0, 1)[frame_index[at:at + n].long()]           # the group's gathered maps
                    outs.append(self.forward(query_points[at:at + n], f, iters, True, down_ratio, is_train, track_feats,
                                             TRACKorPOSE, ind, None if counts is None else counts[at:at + n],
                                             None if frames is None else frames[at:at + n]))
                    at += n
                cat = lambda vs: None if vs[0] is None else torch.cat(vs)  # noqa: E731
                res = ([cat([o[0][i] for o in outs]) for i in range(len(outs[0][0]))],) + tuple(
                    cat([o[k] for o in outs]) for k in range(1, 5))
                return res if return_feat else (res[0], res[1], res[4])
            if frame_index is not None:
                frame_index = frame_index.to(fmaps[0].device)
            group_items = sizes
        else:
            B_items, S_maps = fmaps.shape[:2]
        counts = frames = None
        if num_frames is not None:
            assert not TRACKorPOSE, "num_frames is served with TRACKorPOSE=False only"
            from .utils import check_num_tracks

            frames = check_num_tracks(num_frames, B_items, S_maps)
            live = torch.arange(S_maps, device=query_points.device)[None, :] < torch.tensor(
                frames, device=query_points.device)[:, None]                                  # (B, S)
        if num_tracks is not None:
            assert not TRACKorPOSE, "num_tracks is served with TRACKorPOSE=False only"
            from .utils import check_num_tracks

            counts = check_num_tracks(num_tracks, query_points.shape[0], query_points.shape[1])
            real = torch.arange(query_points.shape[1], device=query_points.device)[None, :] < torch.tensor(
                counts, device=query_points.device)[:, None]                                  # (B, N)
            query_points = query_points * real[:, :, None]          # padded queries start at 0 and never move
        if TRACKorPOSE:
            B, S, N, D = query_points.shape
        else:
            B, N, D = query_points.shape
        S = S_maps
        if not grouped:
            B = fmaps.shape[0]
        assert D == 2
        if down_ratio > 1:  # guards BOTH divisions (SURVEY A.6 i)
            query_points = query_points / float(down_ratio)
            query_points = query_points / float(self.stride)
        if TRACKorPOSE:
            coords = query_points.clone()
        else:
            coords = query_points.clone().reshape(B, 1, N, 2).repeat(1, S, 1, 1)
        if frames is not None:
            coords = coords * live[:, :, None, None]

        if grouped:
            bounds = [sum(group_items[:g]) for g in range(len(fmaps) + 1)]
            query_track_feat = torch.cat([sample_features4d(
                f[:, 0] if frame_index is None else f.flatten(0, 1)[frame_index[r0:r1, 0].long()], coords[r0:r1, 0])
                for f, r0, r1 in zip(fmaps, bounds[:-1], bounds[1:])])
        elif isinstance(fmaps, Upsampled2x):
            # bilinear sample (border) of the 2x-1 up-sampling at p == bilinear sample of its source at p / 2
            query_track_feat = sample_features4d(fmaps.src[:, 0], coords[:, 0] * 0.5)
        else:
            query_track_feat = sample_features4d(fmaps[:, 0], coords[:, 0])
        track_feats = query_track_feat.unsqueeze(1).repeat(1, S, 1, 1)
        coords_backup = coords.clone()

        corr_cls = EfficientCorrBlock if self.efficient_corr else CorrBlock
        if grouped:
            fcorr_fn = [corr_cls(f, num_levels=self.corr_levels, radius=self.corr_radius) for f in fmaps]
        else:
            fcorr_fn = corr_cls(fmaps, num_levels=self.corr_levels, radius=self.corr_radius)
        # sampled_pos_emb depends on coords[:, 0] only, which the loop pins -> computed once, not per iteration
        tokenizer = TrackTokenizer(fcorr_fn, coords[:, 0], self.transformer_dim, num_tracks=counts, num_frames=frames,
                                   frame_index=frame_index, group_items=group_items if grouped else None)

        coord_preds = []
        for _ in range(iters):
            coords = coords.detach()
            x = tokenizer.tokens(coords, track_feats)  # (B, N, S, transformer_dim), one fused kernel

            if counts is None and frames is None:
                delta = self.updateformer(x).reshape(B * N, S, self.latent_dim + 2)
            elif frames is None:
                delta = self.updateformer(x, num_tracks=counts).reshape(B * N, S, self.latent_dim + 2)   # 0 when padded
            else:
                delta = self.updateformer(x, num_tracks=counts, num_frames=frames).reshape(B * N, S, self.latent_dim + 2)
            delta_coords_ = delta[:, :, :2]
            delta_feats_ = delta[:, :, 2:].reshape(B * N * S, self.latent_dim)

            track_feats_ = track_feats.permute(0, 2, 1, 3).reshape(B * N * S, self.latent_dim)
            track_feats_ = self.ffeat_updater(self.norm(delta_feats_)) + track_feats_
            track_feats = track_feats_.reshape(B, N, S, self.latent_dim).permute(0, 2, 1, 3)

            coords = coords + delta_coords_.reshape(B, N, S, 2).permute(0, 2, 1, 3)
            coords[:, 0] = coords_backup[:, 0]
            if down_ratio > 1:
                coord_preds.append(coords * self.stride * down_ratio)
            else:
                coord_preds.append(coords * self.stride)

        if not self.fine:
            vis_e = torch.sigmoid(self.vis_predictor(track_feats.reshape(B * S * N, self.latent_dim)).reshape(B, S, N))
        else:
            vis_e = None
        conf_e = None
        if self.cfg.track_conf:
            conf_e = torch.sigmoid(self.conf_predictor(track_feats.reshape(B * S * N, self.latent_dim)).reshape(B, S, N))
        if counts is not None or frames is not None:
            if counts is None:
                real = torch.ones((B, N), dtype=torch.bool, device=coords.device)
            pad_s = ~real[:, None, :] if frames is None else ~(real[:, None, :] & live[:, :, None])  # (B, 1 or S, N)
            coord_preds = [c.masked_fill(pad_s[..., None], 0.0) for c in coord_preds]
            vis_e = None if vis_e is None else vis_e.masked_fill(pad_s, 0.0)
            conf_e = None if conf_e is None else conf_e.masked_fill(pad_s, 0.0)
            track_feats = track_feats.masked_fill(pad_s[..., None], 0.0)
            query_track_feat = query_track_feat.masked_fill(~real[..., None], 0.0)
        if return_feat:
            return coord_preds, vis_e, track_feats, query_track_feat, conf_e
        return coord_preds, vis_e, conf_e
