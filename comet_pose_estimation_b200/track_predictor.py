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
from .packed_frames import pack_referenced_frames
from .refine_track import ShallowEncoder, _inorm, _ResidualBlock, _resize, inverted_score, refine_track
from .utils import check_clip_frames, check_image_sizes, check_num_tracks, check_query_frames, clip_items


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

    def _encode_frames(self, images):
        """(B,S,3,H,W) -> (B,S,128,h,w): one encoder call over all B*S frames."""
        B, S, C, H, W = images.shape
        fmaps = self._encode_flat(images.reshape(B * S, C, H, W))
        return fmaps.reshape(B, S, -1, fmaps.shape[-2], fmaps.shape[-1])

    def _encode_flat(self, x):
        """(F,3,H,W) frames -> (F,128,h,w) maps, one encoder call."""
        H, W = x.shape[-2:]
        if self.coarse_down_ratio > 1:
            # F.interpolate(scale_factor=1/down_ratio, bilinear, align_corners=True): output size floor(H / down_ratio)
            x = _resize(x, (int(H * (1.0 / self.coarse_down_ratio)), int(W * (1.0 / self.coarse_down_ratio))))
        # NCHW on purpose: the channels-last instance-norm kernel of this library is built for the patch encoder's many tiny
        # planes (one thread per (sample, channel)); at 16 x 64 planes of 256 x 256 it would take 20 ms (measured), the
        # NCHW kernel (one warp per plane) 2.9 ms for the whole encoder (torch ops: 5.5 ms)
        return self.coarse_fnet(x.contiguous())

    def min_image_size(self, fine_tracking: bool = True) -> int:
        """The smallest image height or width ``track`` runs: the coarse maps (side ``int(x / coarse_down_ratio) //
        stride``) need one cell at the deepest of the ``corr_levels`` pyramid levels, and the fine tracker cuts 31x31
        patches.  128 for the shipped configuration (down ratio 2, stride 4, 5 levels: 16x16 maps)."""
        p = self.coarse_predictor
        x = 31 if fine_tracking else 1
        while int(x * (1.0 / self.coarse_down_ratio)) // p.stride < 1 << (p.corr_levels - 1):
            x += 1
        return x

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
                    query_frames=None, image_sizes=None, clip_frames=None):
        """``track`` for B sequences in one call: images (B,S,3,H,W), ``query_points``
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
        (B, N_max) int64.  Query frames all 0 run exactly the path without them.

        Sequences of different image sizes: ``images`` a list of B clips (S_b,3,H_b,W_b), or the padded
        (B,S_max,3,H_max,W_max) with ``image_sizes`` (B, 2) integers (H_b, W_b): sequence b's pixels are
        ``images[b, :S_b, :, :H_b, :W_b]`` and no other pixel is read.  Query points and tracks are in each sequence's
        own pixels, sequence b gets what ``track`` returns for it alone (up to the rounding of the iterated loop), with
        ``num_tracks``, ``num_frames`` and ``query_frames`` as above, and the dict gets ``image_sizes`` (B, 2) int64.
        Sizes below ``min_image_size()`` are refused.  Sequences are ordered into size groups whose frames are packed
        into one buffer (:class:`PackedFrames`); the encoder and the token kernels run once per group, the update
        transformer once over all sequences.  When all sizes are equal the one-size path runs unchanged.

        Clips that share frames of a video: ``images`` the source video (T,3,H,W), or a list of videos (T_v,3,H_v,W_v)
        whose frames are numbered one after another, video 0 first; ``clip_frames`` a list of B 1-D integer tensors or
        sequences (S_b,): clip b is made of the frames with those numbers, in that order (repeats and frames shared
        between clips allowed; all frames of a clip of one size).  The call returns what this call returns for the
        gathered clips ``[flat_frames[clip_frames[b]] for b in range(B)]`` with the same ``query_points``,
        ``num_tracks`` and ``query_frames`` (query frames are clip positions), up to the rounding of the iterated loop:
        the same keys and padding, ``num_frames`` included, and ``image_sizes`` when the sizes differ.  ``num_frames``
        and ``image_sizes``, if given, must agree with the clips.  Each referenced frame is copied once, encoded once and
        prepared into the coarse pyramid once; frames no clip references are never read."""
        videos, clips, sizes, S = self._batch_clips(images, num_frames, image_sizes, clip_frames, fine_tracking)
        B = len(clips)
        frames = [len(c) for c in clips]
        mixed = len(set(sizes)) > 1
        listed = not isinstance(images, torch.Tensor)
        query_points, counts = _padded_queries(query_points, num_tracks, B)
        N = query_points.shape[1]
        qf = [[0] * n for n in counts] if query_frames is None else check_query_frames(query_frames, counts, frames)
        if clip_frames is not None or mixed or any(f != S for f in frames) or any(t for q in qf for t in q):
            packed, clip_ids = pack_referenced_frames(videos, clips)
            out = self._track_clips(packed, clip_ids, query_points, counts, qf, S, coarse_iters, fine_tracking)
        else:
            # a plain batch: one size, every frame real, every query on frame 0
            images = torch.stack(videos) if listed else images[..., :sizes[0][0], :sizes[0][1]]
            fmaps = self._encode_frames(images)
            coarse_list, vis, track_feats, query_feat, conf = self.coarse_predictor(
                query_points=query_points, fmaps=fmaps, iters=coarse_iters, down_ratio=self.coarse_down_ratio,
                is_train=False, return_feat=True, TRACKorPOSE=False, num_tracks=counts)
            coarse = coarse_list[-1]
            out = {"coarse_pred_track_list": coarse_list, "coarse_pred_track": coarse, "vis": vis, "conf": conf}
            real = (torch.arange(N, device=coarse.device)[None, :] < torch.tensor(counts, device=coarse.device)[:, None])
            if fine_tracking:
                refined, score = refine_track(images, self.fine_fnet, self.fine_predictor, coarse, compute_score=True,
                                              num_tracks=counts)
                out["refine_pred_track"] = refined
                out["track_score"] = score
                out["pred_score"] = inverted_score(score) * real[:, None, :]
            else:
                out["refine_pred_track"] = coarse
                out["pred_score"] = torch.ones_like(vis) * real[:, None, :]
        out["num_tracks"] = torch.tensor(counts, dtype=torch.int64)
        if num_frames is not None or listed or clip_frames is not None or mixed:
            out["num_frames"] = torch.tensor(frames, dtype=torch.int64)
        if query_frames is not None:
            out["query_frames"] = torch.zeros((B, N), dtype=torch.int64)
            for b, q in enumerate(qf):
                out["query_frames"][b, :len(q)] = torch.tensor(q, dtype=torch.int64)
        if mixed or (image_sizes is not None and clip_frames is None):
            out["image_sizes"] = torch.tensor(sizes, dtype=torch.int64)
        return out

    def _batch_clips(self, images, num_frames, image_sizes, clip_frames, fine_tracking):
        """``track_batch``'s images, validated -> (videos, clips, sizes, S): V source videos (T_v,3,H_v,W_v) whose frames
        are numbered one after another (views, nothing copied), clip b's frame numbers, clip b's (H_b, W_b), and the
        length of the output frame axis: a padded tensor of one size keeps its S_max, every other form gets max(S_b).
        A list of clips is one video per clip; a padded tensor is the videos ``images[b, :S_b, :, :H_b, :W_b]``."""
        if clip_frames is not None:
            videos = [images] if isinstance(images, torch.Tensor) else list(images)
            assert len(videos) >= 1 and all(isinstance(v, torch.Tensor) and v.dim() == 4 and v.shape[1] == 3 for v in videos), \
                "with clip_frames, images must be a video (T, 3, H, W) or a list of videos (T_v, 3, H_v, W_v)"
            assert len({v.device for v in videos}) == 1, "the videos must be on one device"
            hw_of = [tuple(int(x) for x in v.shape[-2:]) for v in videos for _ in range(v.shape[0])]   # per source frame
            clips = check_clip_frames(clip_frames, len(hw_of))
            sizes = []
            for b, c in enumerate(clips):
                hws = sorted({hw_of[t] for t in c})
                assert len(hws) == 1, f"clip {b} mixes frame sizes {hws}"
                sizes.append(hws[0])
        elif isinstance(images, (list, tuple)):
            videos = list(images)
            sizes = [(int(x.shape[-2]), int(x.shape[-1])) for x in videos]
        else:
            assert images.dim() == 5, "images must be (B, S_max, 3, H_max, W_max)"
            B, S, _, H, W = images.shape
            sizes = [(H, W)] * B if image_sizes is None else check_image_sizes(image_sizes, B)
            assert all(h <= H and w <= W for h, w in sizes), f"image_sizes {sizes} exceed the padded {H}x{W}"
            frames = [S] * B if num_frames is None else check_num_tracks(num_frames, B, S)
            videos = [images[b, :n, :, :h, :w] for b, (n, (h, w)) in enumerate(zip(frames, sizes))]
        if clip_frames is None:
            first = [sum(int(v.shape[0]) for v in videos[:b]) for b in range(len(videos))]
            clips = [list(range(f, f + int(v.shape[0]))) for f, v in zip(first, videos)]
        frames = [len(c) for c in clips]
        sized = clip_frames is not None or image_sizes is not None or len(set(sizes)) > 1
        if not isinstance(images, torch.Tensor) or clip_frames is not None:         # the sizes and lengths are the clips'
            what = "the image lists" if clip_frames is None else "the clips"
            assert num_frames is None or check_num_tracks(num_frames, len(clips), max(frames)) == frames, \
                f"num_frames disagrees with {what}"
            assert image_sizes is None or check_image_sizes(image_sizes, len(clips)) == sizes, \
                f"image_sizes disagrees with {what}"
        if sized:
            assert all(v.dim() == 4 and v.shape[1] == 3 for v in videos), "each clip must be (S_b, 3, H_b, W_b)"
            floor = self.min_image_size(fine_tracking)
            assert all(min(h, w) >= floor for h, w in sizes), \
                f"image_sizes {sizes}: this tracker needs at least {floor}x{floor}"
        one_size = isinstance(images, torch.Tensor) and clip_frames is None and len(set(sizes)) == 1
        return videos, clips, sizes, images.shape[1] if one_size else max(frames)

    def _track_clips(self, packed, clip_ids, query_points, counts, qf, S, coarse_iters, fine_tracking):
        """The batch of clips over a packed source buffer: clip b is made of the packed frames ``clip_ids[b]``, all of one
        size, in any order, with repeats and frames shared between clips.  One item per (clip, query position) of the
        query frames ``qf`` (validated lists), items ordered by size group; each item reads its frames through a row of
        the item table (``clip_items``).  Each group's packed frames are encoded by one call on their zero-copy slice,
        and the coarse predictor gets them as one source pool per group; the fine side reads the packed buffer; results
        are scattered back to (clip, position, track) order, S positions (S >= every clip's length)."""
        B = len(clip_ids)
        frames = [len(c) for c in clip_ids]
        N = query_points.shape[1]
        dev = query_points.device
        group_of_hw = {hw: g for g, (hw, _) in enumerate(packed.groups)}
        group_of = [group_of_hw[tuple(packed.frame_hw[c[0]].tolist())] for c in clip_ids]
        items, pos, fine_index = clip_items(clip_ids, qf, group_of, S)
        item_counts = [len(ns) for _, _, ns in items]
        item_frames = None if all(f == S for f in frames) else [frames[b] for b, _, _ in items]
        group_items = [sum(1 for b, _, _ in items if group_of[b] == g) for g in range(len(packed.groups))]
        # coarse table: rows of group g index group g's packed frames, which are its source pool (1, F_g, C, h, w)
        coarse_index = fine_index - torch.tensor([packed.group_first[group_of[b]] for b, _, _ in items])[:, None]
        fmaps = [self._encode_flat(packed.group(g))[None] for g in range(len(packed.groups))]

        item_b = torch.tensor([b for b, _, ns in items for _ in ns], device=dev)
        item_i = torch.tensor([i for i, (_, _, ns) in enumerate(items) for _ in ns], device=dev)
        item_j = torch.tensor([j for _, _, ns in items for j in range(len(ns))], device=dev)
        item_n = torch.tensor([n for _, _, ns in items for n in ns], device=dev)
        q_items = query_points.new_zeros((len(items), max(item_counts), 2))
        q_items[item_i, item_j] = query_points[item_b, item_n]

        # one size: a single source pool with its table, the call a coarse predictor without size groups also serves
        pools = dict(fmaps=fmaps[0]) if len(fmaps) == 1 else dict(fmaps=fmaps, group_items=group_items)
        coarse_list, vis, track_feats, query_feat, conf = self.coarse_predictor(
            query_points=q_items, iters=coarse_iters, down_ratio=self.coarse_down_ratio, is_train=False, return_feat=True,
            TRACKorPOSE=False, num_tracks=item_counts, num_frames=item_frames, frame_index=coarse_index, **pools)
        coarse = coarse_list[-1]
        Ni = coarse.shape[2]
        out = {"coarse_pred_track_list": coarse_list, "coarse_pred_track": coarse, "vis": vis, "conf": conf}
        real = padded_mask(item_counts, [S] * len(items) if item_frames is None else item_frames, S, Ni, coarse.device)
        if fine_tracking:
            refined, score = refine_track(packed, self.fine_fnet, self.fine_predictor, coarse, compute_score=True,
                                          num_tracks=item_counts, num_frames=item_frames, frame_index=fine_index)
            out["refine_pred_track"] = refined
            out["track_score"] = score
            out["pred_score"] = inverted_score(score) * real if item_frames is None else inverted_score_padded(score, real)
        else:
            out["refine_pred_track"] = coarse
            out["pred_score"] = torch.ones_like(vis) * real

        if Ni == N and [(b, q) for b, q, _ in items] == [(b, 0) for b in range(B)]:
            return out          # the items are the clips in batch order with no position swapped: nothing to scatter
        # position s of item i shows clip position pos[i, s], and the swap is its own inverse
        return {k: _scatter_items(v, pos.to(dev), (item_b, item_n, item_i, item_j), B, S, N) for k, v in out.items()}


def _padded_queries(query_points, num_tracks, B: int):
    """``track_batch``'s query points (a list of B (N_b, 2) tensors, or a padded (B, N_max, 2) tensor with optional
    counts) -> (padded (B, N_max, 2) tensor, validated counts)."""
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
    return query_points, check_num_tracks([N] * B if num_tracks is None else num_tracks, B, N)


def _scatter_items(v, pos_of_frame, idx, B: int, S: int, N: int):
    """An output (B', S, N_cap, ...) of a batch of items -> (B, S, N, ...) in (sequence, frame, track) order: position s
    of item i shows frame ``pos_of_frame[i, s]`` of its sequence, and real track j of item i is track ``item_n`` of
    sequence ``item_b`` (``idx`` = (item_b, item_n, item_i, item_j), one entry per real track).  Lists map per entry."""
    if v is None:
        return None
    if isinstance(v, list):
        return [_scatter_items(x, pos_of_frame, idx, B, S, N) for x in v]
    item_b, item_n, item_i, item_j = idx
    g = pos_of_frame.reshape(pos_of_frame.shape + (1,) * (v.dim() - 2)).expand((-1, -1) + tuple(v.shape[2:]))
    v = v.gather(1, g)                                      # (B', S, N_cap, ...) in each sequence's frame order
    res = v.new_zeros((B, S, N) + tuple(v.shape[3:]))
    res[item_b, :, item_n] = v[item_i, :, item_j]
    return res


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
    the frame axis too when the dict has ``num_frames``; ``query_frames`` is cut to (1, N_b); ``image_sizes`` is
    dropped)."""
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

    return [{k: cut(v, b, n, s) for k, v in out.items() if k not in ("num_tracks", "num_frames", "image_sizes")}
            for b, (n, s) in enumerate(zip(counts, frames))]
