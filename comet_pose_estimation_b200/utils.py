"""Samplers and sin/cos encodings with the reference's names and signatures
(comet/models/utils.py:37-101, :724-974), computed by CUDA kernels."""
from __future__ import annotations

from typing import Tuple, Union

import torch

from . import _lib
from ._dev import f32c, inner_contig, pad_mode, require_cuda, require_no_grad, stream_ptr

lib = _lib.lib


def _device(device=None) -> torch.device:
    if device is None:
        if not torch.cuda.is_available():
            raise _lib.CometB200Error("no CUDA device: the sin/cos tables are produced by CUDA kernels only")
        return torch.device("cuda", torch.cuda.current_device())
    return torch.device(device)


def bilinear_sampler(input, coords, align_corners=True, padding_mode="border"):
    """utils.py:874-939.  (B,C,H,W) @ (B,Ho,Wo,2) -> (B,C,Ho,Wo); (B,C,T,H,W) @ (B,Do,Ho,Wo,3)=(t,x,y) ->
    (B,C,Do,Ho,Wo).  Coordinates in pixel units."""
    sizes = input.shape[2:]
    assert len(sizes) in [2, 3]
    require_cuda(input, "input")
    require_cuda(coords, "coords")
    require_no_grad(input, coords)
    x = f32c(input)
    c = f32c(coords)
    pm = pad_mode(padding_mode)
    with torch.cuda.device(x.device):
        if len(sizes) == 2:
            B, C, H, W = x.shape
            assert c.dim() == 4 and c.shape[0] == B and c.shape[-1] == 2
            Ho, Wo = c.shape[1:3]
            out = torch.empty((B, C, Ho, Wo), dtype=torch.float32, device=x.device)
            _lib.check(lib.comet_bilinear_sampler4d_f32(x.data_ptr(), c.data_ptr(), out.data_ptr(), B, C, H, W, Ho,
                                                        Wo, int(bool(align_corners)), pm, stream_ptr(x.device)))
        else:
            B, C, T, H, W = x.shape
            assert c.dim() == 5 and c.shape[0] == B and c.shape[-1] == 3
            Do, Ho, Wo = c.shape[1:4]
            out = torch.empty((B, C, Do, Ho, Wo), dtype=torch.float32, device=x.device)
            _lib.check(lib.comet_bilinear_sampler5d_f32(x.data_ptr(), c.data_ptr(), out.data_ptr(), B, C, T, H, W,
                                                        Do, Ho, Wo, int(bool(align_corners)), pm,
                                                        stream_ptr(x.device)))
    return out


def sample_features4d(input, coords):
    """utils.py:942-974.  (B,C,H,W) sampled at (B,R,2) -> (B,R,C); border padding, align_corners=True.
    ``input`` may be a batch-strided view (e.g. ``fmaps[:, 0]``) or batch-expanded (stride 0)."""
    require_cuda(input, "input")
    require_cuda(coords, "coords")
    require_no_grad(input, coords)
    B, C, H, W = input.shape
    x = input if input.dtype == torch.float32 else input.float()
    c = inner_contig(coords)
    assert c.dim() == 3 and c.shape[0] == B and c.shape[2] == 2
    R = c.shape[1]
    out = torch.empty((B, R, C), dtype=torch.float32, device=x.device)
    if B and C > 1 and x.stride(1) == 1 and x.stride(3) == C and x.stride(2) == W * C:
        # channels-last view (e.g. fmaps[:, 0] of a channels-last patch-feature tensor): sampled in place
        with torch.cuda.device(x.device):
            _lib.check(lib.comet_sample_features4d_cl_f32(x.data_ptr(), x.stride(0), c.data_ptr(), c.stride(0),
                                                          c.stride(1), out.data_ptr(), B, C, H, W, R,
                                                          stream_ptr(x.device)))
        return out
    if B and C and not (x.stride(3) == 1 and x.stride(2) == W and x.stride(1) == H * W):
        x = x.contiguous()
    with torch.cuda.device(x.device):
        _lib.check(lib.comet_sample_features4d_f32(x.data_ptr(), x.stride(0), c.data_ptr(), c.stride(0), c.stride(1),
                                                   out.data_ptr(), B, C, H, W, R, stream_ptr(x.device)))
    return out


def get_2d_embedding(xy: torch.Tensor, C: int, cat_coords: bool = True) -> torch.Tensor:
    """utils.py:65-101 (dup :835-871).  (B,N,2) -> (B,N,2C[+2])."""
    B, N, D = xy.shape
    assert D == 2
    require_cuda(xy, "xy")
    require_no_grad(xy)
    x = f32c(xy)
    out = torch.empty((B, N, 2 * C + (2 if cat_coords else 0)), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(lib.comet_embed2d_f32(x.data_ptr(), out.data_ptr(), B * N, C, int(bool(cat_coords)),
                                         stream_ptr(x.device)))
    return out


def get_1d_sincos_pos_embed_from_grid(embed_dim: int, pos: torch.Tensor) -> torch.Tensor:
    """utils.py:37-62 (dup :807-832) -> (1, M, D) float32; float64 arithmetic inside the kernel.
    ``pos`` is taken as float32 positions (the reference's grids are float32 ``arange``s)."""
    assert embed_dim % 2 == 0
    if pos.device.type != "cuda":
        pos = pos.to(_device())
    p = f32c(pos).reshape(-1)
    out = torch.empty((1, p.numel(), embed_dim), dtype=torch.float32, device=p.device)
    with torch.cuda.device(p.device):
        _lib.check(lib.comet_sincos1d_from_grid_f32(p.data_ptr(), out.data_ptr(), p.numel(), embed_dim,
                                                    stream_ptr(p.device)))
    return out


def get_2d_sincos_pos_embed_from_grid(embed_dim: int, grid: torch.Tensor) -> torch.Tensor:
    """utils.py:780-804 -> (1, M, D): first half encodes grid[0], second half grid[1]."""
    assert embed_dim % 2 == 0
    a = get_1d_sincos_pos_embed_from_grid(embed_dim // 2, grid[0])
    b = get_1d_sincos_pos_embed_from_grid(embed_dim // 2, grid[1])
    return torch.cat([a, b], dim=2)


def get_2d_sincos_pos_embed(embed_dim: int, grid_size: Union[int, Tuple[int, int]], return_grid=False, device=None):
    """utils.py:724-755 -> (1, D, H, W) float32 on the CUDA device (the reference builds it on the host in
    float64 and uploads it; here one kernel evaluates it in float64 on the device)."""
    if isinstance(grid_size, tuple):
        gh, gw = grid_size
    else:
        gh = gw = grid_size
    assert embed_dim % 2 == 0 and (embed_dim // 2) % 2 == 0
    dev = _device(device)
    out = torch.empty((1, embed_dim, gh, gw), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.comet_sincos2d_f32(out.data_ptr(), embed_dim, gh, gw, stream_ptr(dev)))
    if return_grid:
        ys = torch.arange(gh, dtype=torch.float, device=dev)
        xs = torch.arange(gw, dtype=torch.float, device=dev)
        grid = torch.stack(torch.meshgrid(xs, ys, indexing="xy"), dim=0).reshape(2, 1, gh, gw)
        return out, grid
    return out


def get_1d_sincos_pos_embed(embed_dim: int, length: int, return_grid: bool = False, device=None) -> torch.Tensor:
    """utils.py:758-777 (the time encoding of camera_predictor10.py:365-371) -> (1, length, D)."""
    dev = _device(device)
    grid = torch.arange(length, dtype=torch.float, device=dev)
    pe = get_1d_sincos_pos_embed_from_grid(embed_dim, grid)
    if return_grid:
        return pe, grid.unsqueeze(0)
    return pe


def upsample_bilinear_align_corners(x: torch.Tensor, size) -> torch.Tensor:
    """``F.interpolate(x, size, mode="bilinear", align_corners=True)`` for a 4-D float32 CUDA tensor, contiguous or
    channels-last (the output keeps the input's memory format).  The patch encoder of the fine tracker
    (ShallowEncoder.forward, blocks.py:176-190) spends 90 % of ``refine_track`` in ATen's kernel for this op at 8192
    patches; this one is HBM-bound."""
    require_cuda(x, "x")
    require_no_grad(x)
    assert x.dim() == 4
    N, C, Hi, Wi = x.shape
    Ho, Wo = (size, size) if isinstance(size, int) else tuple(size)
    if x.dtype == torch.bfloat16 and x.is_contiguous():
        out = torch.empty((N, C, Ho, Wo), dtype=torch.bfloat16, device=x.device)
        with torch.cuda.device(x.device):
            _lib.check(lib.comet_upsample_bilinear_ac_bf16(x.data_ptr(), out.data_ptr(), N, C, Hi, Wi, Ho, Wo, stream_ptr(x.device)))
        return out
    x = x if x.dtype == torch.float32 else x.float()
    cl = (C % 4 == 0 and C > 1 and not x.is_contiguous() and x.is_contiguous(memory_format=torch.channels_last)
          and x.data_ptr() % 16 == 0)
    if not cl:
        x = x.contiguous()
    out = torch.empty((N, C, Ho, Wo), dtype=torch.float32, device=x.device,
                      memory_format=torch.channels_last if cl else torch.contiguous_format)
    with torch.cuda.device(x.device):
        _lib.check(lib.comet_upsample_bilinear_ac_f32(x.data_ptr(), out.data_ptr(), N, C, Hi, Wi, Ho, Wo,
                                                      _lib.FMAPS_CHANNEL_LAST if cl else _lib.FMAPS_NCHW,
                                                      stream_ptr(x.device)))
    return out


def instance_norm(x: torch.Tensor, relu: bool = False, eps: float = 1e-5) -> torch.Tensor:
    """``nn.InstanceNorm2d(C)(x)`` (affine=False, no running stats; optionally followed by ReLU) for a 4-D float32 or
    bfloat16 CUDA tensor, contiguous or channels-last (dtype kept; memory format kept except for large bf16 planes)."""
    require_cuda(x, "x")
    require_no_grad(x)
    assert x.dim() == 4
    N, C, H, W = x.shape
    if x.dtype == torch.bfloat16 and (x.is_contiguous() or H * W >= 1024):
        # bf16 in, bf16 out (the encoders under torch.autocast): float32 statistics of the bf16 values, one kernel, no
        # cast passes; NCHW (large channels-last planes are re-laid out: the per-plane kernel reads a plane once)
        x = x.contiguous()
        out = torch.empty_like(x)
        with torch.cuda.device(x.device):
            _lib.check(lib.comet_instance_norm_bf16(x.data_ptr(), out.data_ptr(), N, C, H * W, int(relu), float(eps),
                                                    stream_ptr(x.device)))
        return out
    in_dtype = x.dtype
    x = x if x.dtype == torch.float32 else x.float()
    cl = C > 1 and not x.is_contiguous() and x.is_contiguous(memory_format=torch.channels_last)
    if cl and H * W > 4096 and N * C < 148 * 256:
        # few large planes: the channels-last kernel (one thread per (sample, channel), built for the patch encoder's
        # 262144 planes of <= 256 positions) would serialise over H*W; the NCHW kernel (one CTA per plane) does not
        cl = False
    if not cl:
        x = x.contiguous()
    out = torch.empty_like(x)
    with torch.cuda.device(x.device):
        _lib.check(lib.comet_instance_norm_f32(x.data_ptr(), out.data_ptr(), N, C, H * W,
                                               _lib.FMAPS_CHANNEL_LAST if cl else _lib.FMAPS_NCHW, int(relu), float(eps),
                                               stream_ptr(x.device)))
    return out if in_dtype == torch.float32 else out.to(in_dtype)


def check_num_tracks(num_tracks, B: int, N_max: int) -> list:
    """Per-sequence track counts of a padded batch (a sequence of ints or a 1-D tensor) -> list of B Python ints, each in
    [1, N_max].  Anything else raises AssertionError."""
    if isinstance(num_tracks, torch.Tensor):
        assert num_tracks.dim() == 1, f"num_tracks must be 1-D, got shape {tuple(num_tracks.shape)}"
        vals = [int(v) for v in num_tracks.tolist()]
    else:
        vals = [int(v) for v in num_tracks]
    assert len(vals) == B, f"num_tracks has {len(vals)} entries for a batch of {B} sequences"
    assert all(1 <= v <= N_max for v in vals), f"num_tracks {vals} outside [1, {N_max}]"
    return vals


def check_image_sizes(image_sizes, B: int) -> list:
    """Per-sequence image sizes (a (B, 2) integer tensor or nested sequence of (H, W)) -> list of B (H, W) tuples of
    positive Python ints.  Anything else raises AssertionError."""
    t = image_sizes if isinstance(image_sizes, torch.Tensor) else torch.as_tensor(image_sizes)
    assert t.dim() == 2 and tuple(t.shape) == (B, 2), f"image_sizes must be (B, 2) = ({B}, 2), got shape {tuple(t.shape)}"
    assert not t.is_floating_point() and not t.is_complex() and t.dtype != torch.bool, "image_sizes must be integers"
    vals = [(int(h), int(w)) for h, w in t.tolist()]
    assert all(h >= 1 and w >= 1 for h, w in vals), f"image_sizes {vals} must be positive"
    return vals


def check_query_frames(query_frames, counts, frames) -> list:
    """Per-track query frames of a padded batch -> list of B lists of Python ints (list b has counts[b] entries, each in
    [0, frames[b])).  ``query_frames``: a list of B 1-D tensors / sequences with counts[b] entries, or a padded
    (B, N_max) tensor (entries of padded tracks are ignored).  Anything else raises AssertionError."""
    B = len(counts)
    if isinstance(query_frames, torch.Tensor):
        assert query_frames.dim() == 2 and query_frames.shape[0] == B and query_frames.shape[1] >= max(counts), \
            f"query_frames must be (B, N_max) = ({B}, >= {max(counts)}), got shape {tuple(query_frames.shape)}"
        assert not query_frames.is_floating_point(), "query_frames must be integers"
        rows = query_frames.tolist()
        vals = [[int(t) for t in rows[b][:n]] for b, n in enumerate(counts)]
    else:
        vals = []
        for q in query_frames:
            if isinstance(q, torch.Tensor):
                assert q.dim() == 1 and not q.is_floating_point(), "each query_frames entry must be a 1-D integer tensor"
                q = q.tolist()
            vals.append([int(t) for t in q])
        assert len(vals) == B, f"query_frames has {len(vals)} entries for a batch of {B} sequences"
        assert [len(v) for v in vals] == list(counts), \
            f"query_frames lengths {[len(v) for v in vals]} disagree with the track counts {list(counts)}"
    for b, (v, s) in enumerate(zip(vals, frames)):
        assert all(0 <= t < s for t in v), f"query_frames of sequence {b} outside [0, {s})"
    return vals


def query_frame_items(query_frames, frames, S_max: int):
    """Items of a batch with per-track query frames (validated lists, see ``check_query_frames``): the tracks of
    sequence b with query frame q form item (b, q); items are ordered by (b, q), tracks inside an item keep their order.
    -> (items, frame_index): ``items`` a list of (b, q, track indices); ``frame_index`` (B', S_max) int64 on the CPU,
    entry (i, s) the flat index into the B * S_max source frames of the frame that item i sees at position s: sequence
    b's frames with 0 and q swapped; padded positions s >= frames[b] keep their identity index."""
    items = []
    for b, qf in enumerate(query_frames):
        for q in sorted(set(qf)):
            items.append((b, q, [n for n, t in enumerate(qf) if t == q]))
    frame_index = torch.empty((len(items), S_max), dtype=torch.int64)
    for i, (b, q, _) in enumerate(items):
        order = list(range(S_max))
        order[0], order[q] = q, 0
        frame_index[i] = torch.tensor(order) + b * S_max
    return items, frame_index


def check_clip_frames(clip_frames, num_source_frames: int) -> list:
    """Frame numbers of B clips (a list of B 1-D integer tensors or sequences) -> list of B non-empty lists of Python
    ints, each in [0, num_source_frames).  Anything else raises AssertionError."""
    assert isinstance(clip_frames, (list, tuple)) and len(clip_frames) >= 1, "clip_frames must be a non-empty list of clips"
    vals = []
    for b, c in enumerate(clip_frames):
        t = c if isinstance(c, torch.Tensor) else torch.as_tensor(c)
        assert t.dim() == 1, f"clip {b}: frame numbers must be 1-D, got shape {tuple(t.shape)}"
        assert t.numel() >= 1, f"clip {b} is empty"
        assert not t.is_floating_point() and not t.is_complex() and t.dtype != torch.bool, \
            f"clip {b}: frame numbers must be integers"
        v = [int(x) for x in t.tolist()]
        assert all(0 <= x < num_source_frames for x in v), f"clip {b}: frame numbers outside [0, {num_source_frames})"
        vals.append(v)
    return vals


def clip_items(clip_frames, query_frames, group_of, S=None):
    """Items of a batch of clips over a buffer of source frames: clip b is made of source frames ``clip_frames[b]``
    (validated lists, any order, repeats allowed), and the tracks of clip b with query position q form item (b, q)
    (``query_frames``: validated lists, see ``check_query_frames``).  Items are ordered by (``group_of[b]``, b, q), tracks
    inside an item keep their order; items have S positions (S >= every clip's length; None: the longest clip's).
    -> (items, pos, table), both tables (B', S) int64 on the CPU: ``pos[i, s]`` the clip position that item i shows at
    position s (positions 0 and q swapped; padded positions s >= S_b keep s), and ``table[i, s]`` the source frame
    there, ``clip_frames[b][pos[i, s]]`` (padded positions: the clip's last frame, whose maps are never read)."""
    frames = [len(c) for c in clip_frames]
    S = max(frames) if S is None else S
    items, swapped = query_frame_items(query_frames, frames, S)
    order = sorted(range(len(items)), key=lambda i: group_of[items[i][0]])        # stable: by group, then (b, q)
    items = [items[i] for i in order]
    pos = swapped[order] - torch.tensor([b * S for b, _, _ in items], dtype=torch.int64)[:, None]
    table = torch.tensor([[clip_frames[b][min(p, frames[b] - 1)] for p in row] for (b, _, _), row in zip(items, pos.tolist())],
                         dtype=torch.int64)
    return items, pos, table
