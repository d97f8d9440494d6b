"""Drop-in ``refine_track`` / ``compute_score_fn`` (comet/models/refine_track.py:26-278) and the patch encoder
``ShallowEncoder`` (comet/models/track_modules/blocks.py:114-196) -- the caller of the hot path's second call site
(SURVEY.md section 8f, rank 2/3).

What is B200-specific here is the *data format between the caller and the path*:

* the 31x31 patches are gathered in (b, n, s) order -- the order the fine tracker consumes -- so the reference's
  1 GB ``rearrange("b s n c p q -> (b n) s c p q")`` copy of the encoder output (refine_track.py:122-123) disappears;
* the encoder runs in ``torch.channels_last``; its output, viewed as (B*N, S, C, 31, 31), is the channels-last
  view the fused kernels read zero-copy (one 128-byte line per position: ``_Pyramid.cl_input``).

* the encoder's three bilinear resizes (blocks.py:176-190; the last one, 16x16 -> 31x31, *is* the fine tracker's
  ``fmaps``) run in the library's own kernel: ATen's up-sampling kernel walks batch x channels inside every thread and
  took 192 ms (channels-last) / 314 ms (NCHW) per sequence at 8192 patches on B200 -- 90 % of ``refine_track``;
  with ``comet_upsample_bilinear_ac_f32`` the encoder drops from 207 ms to 13 ms; its instance norms (ATen:
  ``batch_norm`` over N*C "channels", 8.6 ms) run in ``comet_instance_norm_f32`` (+ fused ReLU): 2.4 ms for the
  whole encoder, and ``refine_track`` goes from 226 ms to 26 ms per sequence (``scripts/refine_profile.py``; what
  remains is the torch update transformer).

The convolutions of the encoder (3x3 on 16x16 / 8x8 / 4x4 maps, ~1 ms in cuDNN) stay ``torch.nn`` with the reference's
parameter names.  Results equal the reference's (tests/golden/refine.npz, produced by executing the
reference).
"""
from __future__ import annotations

import torch
import torch.nn as nn
import torch.nn.functional as F

from .blocks import Upsampled2x, up2_supported


# False routes the encoder's resizes / instance norms through the ATen ops even on the GPU (A/B timing in bench.py)
USE_LIBRARY_KERNELS = True
# False makes refine_track materialise the up-sampled patch features (the reference's data flow; A/B timing and tests)
DEFER_UPSAMPLE = True
# False keeps the encoder on the per-operator path (cuDNN convolutions + the library's norm / resize kernels) instead of
# the fused one-kernel encoder (csrc/shallow_encoder.cu); A/B timing and tests
USE_FUSED_ENCODER = True


def _library_ok(x: torch.Tensor) -> bool:
    return (USE_LIBRARY_KERNELS and x.is_cuda and x.dtype in (torch.float32, torch.bfloat16, torch.float16)
            and not (torch.is_grad_enabled() and x.requires_grad))


def _resize(x: torch.Tensor, size) -> torch.Tensor:
    """``F.interpolate(x, size, mode="bilinear", align_corners=True)``.  On the GPU (inference) this is the library's own
    kernel: ATen's up-sampling kernel walks batch x channels inside every thread and, at 8192 patches, is 90 % of
    ``refine_track`` (192-314 ms per sequence on B200 against ~1 ms here).  bf16 / fp16 activations (the encoder under
    ``torch.autocast``) are resized in float32 and cast back -- ATen's path for them is the same slow kernel.  Anything
    else (CPU tensors in the host-logic tests, autograd) takes the torch op."""
    if _library_ok(x):
        from .utils import upsample_bilinear_align_corners

        if x.dtype == torch.float32 or (x.dtype == torch.bfloat16 and x.is_contiguous()):
            return upsample_bilinear_align_corners(x, size)        # (bf16 NCHW: one kernel, bf16 in / bf16 out)
        return upsample_bilinear_align_corners(x.float(), size).to(x.dtype)
    return F.interpolate(x, size, mode="bilinear", align_corners=True)


def _inorm(norm: nn.InstanceNorm2d, x: torch.Tensor, relu: bool) -> torch.Tensor:
    """``relu(norm(x))`` / ``norm(x)``: the library's instance-norm kernel for CUDA inference (ATen routes
    InstanceNorm2d through batch_norm over N*C channels: 8.6 ms per sequence at 8192 patches), torch otherwise."""
    if _library_ok(x):
        from .utils import instance_norm

        return instance_norm(x, relu=relu, eps=norm.eps)      # dtype kept; bf16 (autocast) large planes: one bf16 kernel
    y = norm(x)
    return F.relu(y) if relu else y


class _ResidualBlock(nn.Module):
    """comet/models/modules.py:39-117 with norm_fn="instance" (parameter-free norms); parameter names kept."""

    def __init__(self, in_planes: int, planes: int, stride: int = 1):
        super().__init__()
        self.conv1 = nn.Conv2d(in_planes, planes, kernel_size=3, padding=1, stride=stride)
        self.conv2 = nn.Conv2d(planes, planes, kernel_size=3, padding=1)
        self.norm1 = nn.InstanceNorm2d(planes)
        self.norm2 = nn.InstanceNorm2d(planes)
        if stride == 1:
            self.downsample = None
        else:
            self.norm3 = nn.InstanceNorm2d(planes)
            self.downsample = nn.Sequential(nn.Conv2d(in_planes, planes, kernel_size=1, stride=stride), self.norm3)

    def forward(self, x):
        y = _inorm(self.norm1, self.conv1(x), True)
        y = _inorm(self.norm2, self.conv2(y), True)
        if self.downsample is not None:
            x = _inorm(self.norm3, self.downsample[0](x), False)
        return F.relu(x + y)


class ShallowEncoder(nn.Module):
    """blocks.py:114-196 (``norm_fn="instance"``, the shipped configuration): state-dict keys ``conv1.*``,
    ``layer1.{conv1,conv2,downsample.0}.*``, ``layer2.*``, ``conv2.*``."""

    def __init__(self, input_dim=3, output_dim=32, stride=1, norm_fn="instance", cfg=None):
        super().__init__()
        if norm_fn != "instance":
            raise NotImplementedError("only the shipped norm_fn='instance' configuration is mirrored")
        self.stride = stride
        self.norm_fn = norm_fn
        self.in_planes = output_dim
        self.norm1 = nn.InstanceNorm2d(output_dim)
        self.norm2 = nn.InstanceNorm2d(output_dim * 2)  # constructed by the reference, never used
        self.conv1 = nn.Conv2d(input_dim, output_dim, kernel_size=3, stride=2, padding=1)
        self.layer1 = _ResidualBlock(output_dim, output_dim, stride=2)
        self.layer2 = _ResidualBlock(output_dim, output_dim, stride=2)
        self.conv2 = nn.Conv2d(output_dim, output_dim, kernel_size=1)
        for m in self.modules():
            if isinstance(m, nn.Conv2d):
                nn.init.kaiming_normal_(m.weight, mode="fan_out", nonlinearity="relu")

    _PARAM_ORDER = ("conv1", "layer1.conv1", "layer1.conv2", "layer1.downsample.0",
                    "layer2.conv1", "layer2.conv2", "layer2.downsample.0", "conv2")

    def _fused_ok(self, x: torch.Tensor, H: int, W: int) -> bool:
        """The one-kernel encoder (csrc/shallow_encoder.cu) covers the shipped configuration: 3 -> 32 channels, stride 1,
        31x31 patches, float32 parameters, CUDA inference.  Everything else takes the per-operator path below."""
        w = self.conv1.weight
        return (USE_FUSED_ENCODER and USE_LIBRARY_KERNELS and x.is_cuda and x.dtype == torch.float32 and (H, W) == (31, 31)
                and tuple(w.shape) == (32, 3, 3, 3) and self.stride == 1 and w.dtype == torch.float32 and w.device == x.device
                and not (torch.is_grad_enabled() and (x.requires_grad or w.requires_grad)))

    def packed_parameters(self) -> torch.Tensor:
        """The 16 state-dict tensors in the layout the fused kernel reads (``comet_shallow_encoder_pack_f32``); rebuilt
        when a parameter is replaced or modified in place."""
        mods = [self.get_submodule(n) for n in self._PARAM_ORDER]
        tensors = [t for m in mods for t in (m.weight, m.bias)]
        key = tuple((t.data_ptr(), t._version) for t in tensors)
        cache = getattr(self, "_packed_cache", None)
        if cache is None or cache[0] != key:
            import ctypes

            from . import _lib
            from ._dev import stream_ptr

            dev = tensors[0].device
            keep = [t.detach().contiguous() for t in tensors]
            packed = torch.empty(int(_lib.lib.comet_shallow_encoder_packed_elems()), dtype=torch.float32, device=dev)
            ptrs = (ctypes.c_void_p * 16)(*[t.data_ptr() for t in keep])
            with torch.cuda.device(dev):
                _lib.check(_lib.lib.comet_shallow_encoder_pack_f32(ptrs, packed.data_ptr(), stream_ptr(dev)))
            cache = (key, packed)
            object.__setattr__(self, "_packed_cache", cache)
        return cache[1]

    def _fused_result(self, half_cl: torch.Tensor, size, defer_upsample: bool):
        half = half_cl.permute(0, 3, 1, 2)   # (P, 32, 16, 16) shape, channels-last memory
        if defer_upsample:
            return half, size
        return _resize(half, size)

    def encode_patches_of(self, images: torch.Tensor, topleft: torch.Tensor, defer_upsample: bool = True):
        """``forward(extract_patches(images, topleft, 31))`` without the patch tensor: the kernel reads patch (b, n, s)
        straight from ``images`` (B,S,3,H,W) at the clamped integer corners ``topleft`` (B,S,N,2)."""
        from . import _lib
        from ._dev import stream_ptr

        B, S, _, H, W = images.shape
        N = topleft.shape[2]
        img = images.contiguous()
        tl32 = topleft.to(torch.int32).contiguous()
        out = torch.empty((B * N * S, 16, 16, 32), dtype=torch.float32, device=images.device)
        with torch.cuda.device(images.device):
            _lib.check(_lib.lib.comet_shallow_encoder_from_images_f32(
                img.data_ptr(), tl32.data_ptr(), self.packed_parameters().data_ptr(), out.data_ptr(), B, S, N, H, W,
                float(self.norm1.eps), stream_ptr(images.device)))
        return self._fused_result(out, (31 // self.stride, 31 // self.stride), defer_upsample)

    def encode_packed_patches_of(self, images: torch.Tensor, topleft: torch.Tensor, seq_of_track: torch.Tensor,
                                 defer_upsample: bool = True, num_frames: torch.Tensor = None,
                                 frame_index: torch.Tensor = None):
        """``encode_patches_of`` for P tracks packed from the sequences of ``images`` (B,S,3,H,W): ``topleft`` (P,S,2)
        corners, ``seq_of_track`` (P,) the sequence of each track.  Maps in (track, frame) order, each one bit-identical
        to ``encode_patches_of`` on the same patch.  ``num_frames`` (B,) int32 on the device, or None: sequence b has
        num_frames[b] real frames; the pixels of the other frames are never read and their maps are zeros.

        ``frame_index`` (B', S) integer tensor on the device: the tracks belong to B' items (``seq_of_track`` and
        ``num_frames`` index items) and frame s of item i is image frame ``frame_index[i, s]`` of the B * S_src frames of
        ``images`` (B, S_src, 3, H, W), any S_src; a frame may be read by any number of (item, position) entries."""
        from . import _lib
        from ._dev import stream_ptr

        B, S_src, _, H, W = images.shape
        P, S = topleft.shape[:2]
        assert frame_index is not None or S_src == S, "images and corners disagree on the frame count"
        img = images.contiguous()
        tl32 = topleft.to(torch.int32).contiguous()
        seq32 = seq_of_track.to(device=images.device, dtype=torch.int32).contiguous()
        out = torch.empty((P * S, 16, 16, 32), dtype=torch.float32, device=images.device)
        with torch.cuda.device(images.device):
            if frame_index is not None:
                nf32 = None if num_frames is None else num_frames.to(device=images.device, dtype=torch.int32).contiguous()
                fi32 = frame_index.to(device=images.device, dtype=torch.int32).contiguous()
                _lib.check(_lib.lib.comet_shallow_encoder_from_images_indexed_f32(
                    img.data_ptr(), tl32.data_ptr(), seq32.data_ptr(), None if nf32 is None else nf32.data_ptr(),
                    fi32.data_ptr(), B * S_src, self.packed_parameters().data_ptr(), out.data_ptr(), P, fi32.shape[0], S, H, W,
                    float(self.norm1.eps), stream_ptr(images.device)))
            elif num_frames is None:
                _lib.check(_lib.lib.comet_shallow_encoder_from_images_ragged_f32(
                    img.data_ptr(), tl32.data_ptr(), seq32.data_ptr(), self.packed_parameters().data_ptr(), out.data_ptr(), P,
                    B, S, H, W, float(self.norm1.eps), stream_ptr(images.device)))
            else:
                nf32 = num_frames.to(device=images.device, dtype=torch.int32).contiguous()
                _lib.check(_lib.lib.comet_shallow_encoder_from_images_varlen_f32(
                    img.data_ptr(), tl32.data_ptr(), seq32.data_ptr(), nf32.data_ptr(), self.packed_parameters().data_ptr(),
                    out.data_ptr(), P, B, S, H, W, float(self.norm1.eps), stream_ptr(images.device)))
        return self._fused_result(out, (31 // self.stride, 31 // self.stride), defer_upsample)

    def encode_packed_frames_patches_of(self, frames, topleft: torch.Tensor, seq_of_track: torch.Tensor,
                                        defer_upsample: bool = True, num_frames: torch.Tensor = None,
                                        frame_index: torch.Tensor = None):
        """``encode_packed_patches_of`` reading a :class:`PackedFrames` buffer of frames with different sizes: frame s of
        item ``seq_of_track[p]`` is packed frame ``frame_index[item, s]`` ((B', S) integer tensor on the device; None:
        item * S + s).  Each corner is clamped to its own frame.  Each map is bit-identical to
        ``encode_packed_patches_of`` on an image tensor holding that frame."""
        from . import _lib
        from ._dev import stream_ptr

        dev = frames.device
        P, S = topleft.shape[:2]
        tl32 = topleft.to(torch.int32).contiguous()
        seq32 = seq_of_track.to(device=dev, dtype=torch.int32).contiguous()
        nf32 = None if num_frames is None else num_frames.to(device=dev, dtype=torch.int32).contiguous()
        fi32 = None if frame_index is None else frame_index.to(device=dev, dtype=torch.int32).contiguous()
        B_items = fi32.shape[0] if fi32 is not None else (int(seq32.max()) + 1 if P else 1)
        offsets, hw = frames.device_tables()
        out = torch.empty((P * S, 16, 16, 32), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            _lib.check(_lib.lib.comet_shallow_encoder_from_images_packed_f32(
                frames.data.data_ptr(), offsets.data_ptr(), hw.data_ptr(), frames.num_frames, tl32.data_ptr(),
                seq32.data_ptr(), None if nf32 is None else nf32.data_ptr(), None if fi32 is None else fi32.data_ptr(),
                self.packed_parameters().data_ptr(), out.data_ptr(), P, B_items, S, float(self.norm1.eps), stream_ptr(dev)))
        return self._fused_result(out, (31 // self.stride, 31 // self.stride), defer_upsample)

    def forward(self, x, defer_upsample: bool = False):
        """``defer_upsample=True`` returns the map *before* the last resize together with the size that resize would
        produce -- ``(x_half, (Ho, Wo))`` -- for callers that consume the up-sampling lazily (:class:`Upsampled2x`)."""
        _, _, H, W = x.shape
        if self._fused_ok(x, H, W):
            from . import _lib
            from ._dev import stream_ptr

            P = x.shape[0]
            out = torch.empty((P, 16, 16, 32), dtype=torch.float32, device=x.device)
            sn, sc, sy, sx = x.stride()
            with torch.cuda.device(x.device):
                _lib.check(_lib.lib.comet_shallow_encoder_f32(x.data_ptr(), sn, sc, sy, sx, self.packed_parameters().data_ptr(),
                                                              out.data_ptr(), P, float(self.norm1.eps), stream_ptr(x.device)))
            return self._fused_result(out, (H // self.stride, W // self.stride), defer_upsample)
        x = _inorm(self.norm1, self.conv1(x), True)
        tmp = self.layer1(x)
        x = x + _resize(tmp, x.shape[-2:])
        tmp = self.layer2(tmp)
        x = x + _resize(tmp, x.shape[-2:])
        x = self.conv2(x) + x
        size = (H // self.stride, W // self.stride)
        if defer_upsample:
            return x, size
        return _resize(x, size)


def extract_patches(images: torch.Tensor, topleft: torch.Tensor, psize: int) -> torch.Tensor:
    """``images`` (B,S,C,H,W), ``topleft`` (B,S,N,2) integer (x, y) corners -> patches (B*N*S, C, psize, psize) in
    (b, n, s) order, channels-last memory format.  Same pixels as the reference's unfold + advanced indexing
    (refine_track.py:71-111) without the (B*S, N, C, p, p) intermediate in (s, n) order.  Corners outside
    [0, W-psize] x [0, H-psize] are clamped to it (the reference's indexing would raise IndexError)."""
    B, S, C, H, W = images.shape
    N = topleft.shape[2]
    dev = images.device
    assert H >= psize and W >= psize, "images smaller than the patch"
    topleft = torch.stack([topleft[..., 0].clamp(0, W - psize), topleft[..., 1].clamp(0, H - psize)], dim=-1)
    if USE_LIBRARY_KERNELS and images.is_cuda and images.dtype == torch.float32:
        from . import _lib
        from ._dev import stream_ptr

        img = images.contiguous()
        tl32 = topleft.to(torch.int32).contiguous()
        out = torch.empty((B * N * S, psize, psize, C), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            _lib.check(_lib.lib.comet_extract_patches_f32(img.data_ptr(), tl32.data_ptr(), out.data_ptr(), B, S, N, C, H, W,
                                                          psize, stream_ptr(dev)))
        return out.permute(0, 3, 1, 2)  # NCHW shape, NHWC memory
    ar = torch.arange(psize, device=dev)
    tl = topleft.permute(0, 2, 1, 3).long()                       # (B,N,S,2)
    ys = tl[..., 1, None] + ar                                    # (B,N,S,p)
    xs = tl[..., 0, None] + ar
    bi = torch.arange(B, device=dev).view(B, 1, 1, 1, 1)
    si = torch.arange(S, device=dev).view(1, 1, S, 1, 1)
    img = images.permute(0, 1, 3, 4, 2)                            # (B,S,H,W,C) view
    patches = img[bi, si, ys[..., :, None], xs[..., None, :]]     # (B,N,S,p,p,C)
    return patches.reshape(B * N * S, psize, psize, C).permute(0, 3, 1, 2)  # NCHW shape, NHWC memory


def refine_track(images, fine_fnet, fine_tracker, coarse_pred, pradius=15, sradius=2, compute_score=False,
                 num_tracks=None, num_frames=None, frame_index=None):
    """refine_track.py:26-171.  ``images`` (B,S,3,H,W); ``coarse_pred`` (B,S,N,2) pixels ->
    (refined_tracks (B,S,N,2), score (B,S,N) | None).

    ``num_tracks`` (B ints or a 1-D tensor): ``coarse_pred`` is a padded batch; sequence b's tracks get what the call on
    that sequence alone returns (including the score quirk as it behaves for one sequence: every window of sequence b
    is cut from the frame-0 map of its own first track), entries of padded tracks are 0.  ``num_frames`` (likewise):
    sequence b has the first ``num_frames[b]`` frames; the images of the others are never read and their entries are 0.

    ``frame_index`` ((B', S) integer tensor): ``coarse_pred`` (B', S, N, 2) is a batch of items that read the frames of
    ``images`` (B_src, S_src, 3, H, W), any S_src, in their own order -- item i's frame s is image frame
    ``frame_index[i, s]`` of the B_src * S_src frames, and a frame may be read by any number of items and positions --
    and ``num_tracks`` / ``num_frames`` count per item.  The result is the call on the gathered
    images ``images.flatten(0, 1)[frame_index]``; the patch encoder reads through the table, nothing is gathered.

    ``images`` a :class:`PackedFrames` buffer (frames of different sizes; ``frame_index`` required): item i's frame s is
    packed frame ``frame_index[i, s]``, and every frame of an item has the item's size.  Each track's patch corners are
    clamped to its own item's (W, H); everything after the patch encoder does not depend on the image size."""
    from .packed_frames import PackedFrames

    packed = isinstance(images, PackedFrames)
    if num_tracks is not None or num_frames is not None or frame_index is not None or packed:
        from .utils import check_num_tracks

        B, S, N = coarse_pred.shape[:3]
        counts = check_num_tracks([N] * B if num_tracks is None else num_tracks, B, N)
        frames = None if num_frames is None else check_num_tracks(num_frames, B, S)
        assert not packed or frame_index is not None, "packed frames are read through frame_index"
        if frame_index is not None:
            assert frame_index.dim() == 2 and tuple(frame_index.shape) == (B, S), \
                f"frame_index must be (B', S) = ({B}, {S})"
        return _refine_track_ragged(images, fine_fnet, fine_tracker, coarse_pred, pradius, sradius, compute_score, counts,
                                    frames, frame_index)
    B, S, N, _ = coarse_pred.shape
    _, _, _, H, W = images.shape
    psize = pradius * 2 + 1
    query_points = coarse_pred[:, 0]

    track_int = coarse_pred.floor().int()
    track_frac = coarse_pred - track_int
    topleft = track_int - pradius
    topleft_BSN = topleft.clone()
    # the reference clamps both axes with H - psize (refine_track.py:93-96: it assumes H == W and raises IndexError
    # otherwise); clamping x with W and y with H is the same for square images and stays in bounds for the others
    topleft = torch.stack([topleft[..., 0].clamp(0, W - psize), topleft[..., 1].clamp(0, H - psize)], dim=-1)

    patch_feat = None
    from .base_track_predictor import BaseTrackerPredictor

    lazy = (USE_LIBRARY_KERNELS and DEFER_UPSAMPLE and isinstance(fine_fnet, ShallowEncoder) and images.is_cuda
            and isinstance(fine_tracker, BaseTrackerPredictor) and not torch.is_grad_enabled())
    # one kernel from the images to the encoder's 16x16 map: the patches themselves are never written either
    from_images = lazy and images.shape[2] == 3 and psize == 31 and fine_fnet._fused_ok(images, psize, psize)
    patch_input = None
    if not from_images:
        with torch.no_grad():
            patch_input = extract_patches(images, topleft, psize)
    if lazy:
        # The encoder's last op is an exact 2x-1 bilinear up-sampling (16x16 -> 31x31): hand the fine tracker the
        # half-resolution map and let the fused lookup evaluate the up-sampled pyramid from it (blocks.Upsampled2x) --
        # the 1 GB-per-sequence patch-feature tensor is never written.
        if from_images:
            half, size = fine_fnet.encode_patches_of(images, topleft, defer_upsample=True)
        else:
            half, size = fine_fnet(patch_input, defer_upsample=True)
        Hs, Ws = half.shape[-2:]
        if size == (2 * Hs - 1, 2 * Ws - 1) and size == (psize, psize):
            C_out = half.shape[1]
            half = half.contiguous(memory_format=torch.channels_last)
            # (B*N*S, C, Hs, Ws) channels-last memory == (B*N, S, Hs, Ws, C): the (b n) s c p q view, no copy
            src = half.permute(0, 2, 3, 1).reshape(B * N, S, Hs, Ws, C_out).permute(0, 1, 4, 2, 3)
            up = Upsampled2x(src)
            if up2_supported(up, fine_tracker.corr_levels, fine_tracker.corr_radius, "zeros") and not fine_tracker.efficient_corr:
                patch_feat = up
            else:
                patch_feat = _resize(half, size)
        else:
            patch_feat = _resize(half, size)
    if patch_feat is None:
        patch_feat = fine_fnet(patch_input)                        # (B*N*S, C_out, p, p), channels-last memory
    if not isinstance(patch_feat, Upsampled2x):
        C_out = patch_feat.shape[1]
        patch_feat = patch_feat.reshape(B * N, S, C_out, psize, psize)  # a view: (b n) s c p q, no rearrange copy

    patch_query_points = (track_frac[:, 0] + pradius).reshape(B * N, 2).unsqueeze(1)
    fine_pred_track_lists, _, _, query_point_feat, _ = fine_tracker(
        query_points=patch_query_points, fmaps=patch_feat, iters=6, return_feat=True, TRACKorPOSE=False)
    fine_pred_track = fine_pred_track_lists[-1].clone()            # (B*N, S, 1, 2), relative to the patch corner

    for idx in range(len(fine_pred_track_lists)):
        lvl = fine_pred_track_lists[idx].reshape(B, N, S, 1, 2).permute(0, 2, 1, 3, 4).squeeze(-2)
        fine_pred_track_lists[idx] = lvl + topleft_BSN
    refined_tracks = fine_pred_track_lists[-1].clone()
    refined_tracks[:, 0] = query_points

    score = None
    if compute_score:
        score = compute_score_fn(query_point_feat, patch_feat, fine_pred_track, sradius, psize, B, N, S, C_out)
    return refined_tracks, score


def _refine_track_ragged(images, fine_fnet, fine_tracker, coarse_pred, pradius, sradius, compute_score, counts, frames=None,
                         frame_index=None):
    """The fine tracker works per track, so the real tracks of all sequences run as ONE packed batch of P = sum(counts)
    tracks, without per-sequence padding: the fused encoder reads each track's patches from its own sequence's frames.  Configurations
    without the fused encoder run the per-sequence definition.  ``frames``: per-sequence frame counts (None: all S); each
    packed track then runs its own sequence's frame count through the fine tracker.  ``frame_index``: the sequences are
    items reading the frames of ``images`` through the table (see ``refine_track``); ``images`` may be a
    :class:`PackedFrames` buffer."""
    from .base_track_predictor import BaseTrackerPredictor
    from .packed_frames import PackedFrames

    B, S, N, _ = coarse_pred.shape
    packed = images if isinstance(images, PackedFrames) else None
    pix = images if packed is None else packed.data
    psize = pradius * 2 + 1
    dev = coarse_pred.device
    fused = (USE_LIBRARY_KERNELS and DEFER_UPSAMPLE and isinstance(fine_fnet, ShallowEncoder) and pix.is_cuda
             and isinstance(fine_tracker, BaseTrackerPredictor) and not torch.is_grad_enabled()
             and (packed is not None or images.shape[2] == 3) and psize == 31 and fine_fnet._fused_ok(pix, psize, psize))
    if not fused:
        if packed is not None:
            fi_host = frame_index.tolist()
        elif frame_index is not None:
            images = images.flatten(0, 1)[frame_index.to(images.device).long()]          # (B', S, 3, H, W)
        refined = coarse_pred.new_zeros(coarse_pred.shape)
        score = coarse_pred.new_zeros((B, S, N)) if compute_score else None
        for b, n in enumerate(counts):
            sb = S if frames is None else frames[b]
            img = images[b:b + 1, :sb] if packed is None else torch.cat([packed.frames(f, 1) for f in fi_host[b][:sb]])[None]
            r, sc = refine_track(img, fine_fnet, fine_tracker, coarse_pred[b:b + 1, :sb, :n], pradius, sradius,
                                 compute_score)
            refined[b, :sb, :n] = r[0]
            if compute_score:
                score[b, :sb, :n] = sc[0]
        return refined, score

    # The packed count is rounded up to one of four buckets per octave, so that the fine transformer's captured graphs
    # (keyed by shape) serve a dataset's changing counts; the padding tracks read sequence 0 at corner 0 and are dropped.
    P = sum(counts)
    quantum = 1 << max(P.bit_length() - 3, 0)
    P_cap = (P + quantum - 1) // quantum * quantum
    seq_host = [b for b, n in enumerate(counts) for _ in range(n)]
    seq_real = torch.tensor(seq_host, device=dev)                          # (P,) sequence of each packed track
    loc = torch.tensor([j for n in counts for j in range(n)], device=dev)  # (P,) its index inside the sequence
    first = torch.tensor([sum(counts[:b]) for b in range(B)], device=dev)  # (B,) packed index of each first track
    seq = torch.cat([seq_real, seq_real.new_zeros(P_cap - P)])
    coarse = torch.cat([coarse_pred[seq_real, :, loc], coarse_pred.new_zeros((P_cap - P, S, 2))])   # (P_cap, S, 2)
    query_points = coarse[:, 0]
    track_int = coarse.floor().int()
    track_frac = coarse - track_int
    topleft_raw = track_int - pradius
    dev_frames = None if frames is None else torch.tensor(frames, dtype=torch.int32, device=dev)
    if packed is None:
        _, _, _, H, W = images.shape
        topleft = torch.stack([topleft_raw[..., 0].clamp(0, W - psize), topleft_raw[..., 1].clamp(0, H - psize)], dim=-1)
        half, size = fine_fnet.encode_packed_patches_of(images, topleft, seq, defer_upsample=True, num_frames=dev_frames,
                                                        frame_index=None if frame_index is None else frame_index.to(dev))
    else:
        # every frame of an item has the item's size: each track is clamped to its own item's (W, H)
        hw = packed.frame_hw[frame_index[:, 0].cpu().long()].to(dev)[seq]                # (P_cap, 2) = (H, W)
        topleft = torch.stack([torch.minimum(topleft_raw[..., 0].clamp(min=0), hw[:, 1:2] - psize),
                               torch.minimum(topleft_raw[..., 1].clamp(min=0), hw[:, 0:1] - psize)], dim=-1)
        half, size = fine_fnet.encode_packed_frames_patches_of(packed, topleft, seq, defer_upsample=True,
                                                               num_frames=dev_frames, frame_index=frame_index.to(dev))
    Hs, Ws = half.shape[-2:]
    C_out = half.shape[1]
    half = half.contiguous(memory_format=torch.channels_last)
    patch_feat = None
    if size == (2 * Hs - 1, 2 * Ws - 1) and size == (psize, psize):
        src = half.permute(0, 2, 3, 1).reshape(P_cap, S, Hs, Ws, C_out).permute(0, 1, 4, 2, 3)
        up = Upsampled2x(src)
        if up2_supported(up, fine_tracker.corr_levels, fine_tracker.corr_radius, "zeros") and not fine_tracker.efficient_corr:
            patch_feat = up
    if patch_feat is None:
        patch_feat = _resize(half, size).reshape(P_cap, S, C_out, psize, psize)

    patch_query_points = (track_frac[:, 0] + pradius).reshape(P_cap, 2).unsqueeze(1)
    if frames is None:
        fine_lists, _, _, query_point_feat, _ = fine_tracker(
            query_points=patch_query_points, fmaps=patch_feat, iters=6, return_feat=True, TRACKorPOSE=False)
    else:
        fine_lists, _, _, query_point_feat, _ = fine_tracker(
            query_points=patch_query_points, fmaps=patch_feat, iters=6, return_feat=True, TRACKorPOSE=False,
            num_frames=dev_frames[seq])
    fine_pred_track = fine_lists[-1][:P].clone()                           # (P, S, 1, 2), relative to the patch corner
    refined_p = fine_lists[-1][:P].squeeze(-2) + topleft_raw[:P]           # (P, S, 2)
    refined_p[:, 0] = query_points[:P]
    if frames is not None:
        refined_p = refined_p.masked_fill((torch.arange(S, device=dev)[None, :] >= dev_frames[seq_real][:, None])[..., None],
                                          0.0)
    refined = coarse_pred.new_zeros(coarse_pred.shape)
    refined[seq_real, :, loc] = refined_p

    score = None
    if compute_score:
        score = _score_ragged(query_point_feat[:P].reshape(P, C_out), patch_feat, fine_pred_track, sradius, psize, counts,
                              first, B, N, S, C_out, frames)
    return refined, score


def _score_ragged(query_point_feat, patch_feat, fine_pred_track, sradius, psize, counts, first, B, N, S, C_out,
                  frames=None):
    """``compute_score_fn`` of every sequence of a packed batch at once, each as the single-sequence call computes it:
    its windows cut from the frame-0 map of its first track, at the corners of its own k-th track in (n, s) order re-read
    as (s, n), with the sequence's own frame count as S.  -> (B, S, N), zeros for padded tracks and frames."""
    dev = fine_pred_track.device
    ssize = sradius * 2 + 1
    cnt = torch.tensor(counts, device=dev)
    frm = torch.tensor([S] * B if frames is None else frames, device=dev)
    corner = (fine_pred_track.floor().int() - sradius).clamp(0, psize - ssize).squeeze(2)   # (P, S, 2) = (x, y)
    bb = torch.arange(B, device=dev)[:, None, None].expand(B, S - 1, N)
    sp = torch.arange(1, S, device=dev)[None, :, None].expand(B, S - 1, N)
    nn_ = torch.arange(N, device=dev)[None, None, :].expand(B, S - 1, N)
    nb, sb = cnt[bb], frm[bb]
    real = (nn_ < nb) & (sp < sb)
    k = sp * nb + nn_                                   # position (s, n) of sequence b reads window k of its (n, s) list
    src_track = torch.where(real, first[bb] + k // sb, first[bb])
    src_frame = torch.where(real, k % sb, torch.zeros_like(k))
    b_r, src_track, src_frame = bb[real], src_track[real], src_frame[real]
    q = query_point_feat[first[b_r] + nn_[real]]       # (M, C)
    cx = corner[src_track, src_frame, 0].long()
    cy = corner[src_track, src_frame, 1].long()
    ar = torch.arange(ssize, device=dev)
    rows = (cy[:, None] + ar)[:, :, None]
    cols = (cx[:, None] + ar)[:, None, :]
    if isinstance(patch_feat, Upsampled2x):
        small = patch_feat.materialize(first * S)                                         # (B, C, p, p)
    else:
        small = patch_feat[first, 0]
    win = small[b_r[:, None, None], :, rows, cols]                                        # (M, ss, ss, C)
    win = win.permute(0, 3, 1, 2).reshape(-1, C_out, ssize * ssize)
    sim = torch.einsum("mc,mcr->mr", q, win)
    heat = torch.softmax(sim * (1.0 / C_out ** 0.5), dim=1)
    lin = torch.linspace(-1.0, 1.0, ssize, device=heat.device, dtype=heat.dtype)
    grid = torch.stack([lin.repeat(ssize), lin.repeat_interleave(ssize)], -1)
    mean = heat @ grid
    var = heat @ (grid ** 2) - mean ** 2
    std = torch.sqrt(torch.clamp(var, min=1e-10)).sum(-1)
    score = std.new_zeros((B, S, N))
    score[:, 1:][real] = std
    score[:, 0] = (torch.arange(N, device=dev)[None, :] < cnt[:, None]).to(score.dtype)
    return score


def inverted_score(track_score: torch.Tensor, eps: float = 1e-6) -> torch.Tensor:
    """``COMET.forward_all``'s conversion of the fine tracker's score into the track confidence the camera predictor
    consumes (E2Epose2.py:232-236): ``1 / (score + eps)`` normalised by its maximum over the frames of each track."""
    inv = 1.0 / (track_score + eps)
    return inv / inv.max(dim=1, keepdim=True)[0]


def compute_score_fn(query_point_feat, patch_feat, fine_pred_track, sradius, psize, B, N, S, C_out):
    """refine_track.py:174-278: std of the softmax similarity heat-map of the query feature against a
    (2*sradius+1)^2 window of patch features.  Reproduces the reference's indexing exactly, including its quirk
    (SURVEY.md A.6 iii): the k-th window is cut from patch map number ``b`` of the (b s n)-ordered list -- for
    B == 1 always map 0 -- at the corner of the k-th track in (b n, s) order, then the list is re-read as (b, s, n)."""
    ssize = sradius * 2 + 1
    M = B * S * N
    q = query_point_feat.reshape(B, N, C_out).unsqueeze(1).expand(-1, S - 1, -1, -1).reshape(B * (S - 1) * N, C_out)

    corner = (fine_pred_track.floor().int() - sradius).clamp(0, psize - ssize).squeeze(2)   # (B*N, S, 2) = (x, y)
    cx = corner[..., 0].flatten().long()          # k runs over (b n, s)
    cy = corner[..., 1].flatten().long()
    which = torch.arange(B, device=patch_feat.device)[:, None, None].expand(-1, S, N).reshape(-1)  # k over (b, s, n)

    # map m of the (b s n)-ordered list = patch_feat[b*N + n, s]
    m = which
    mb, ms, mn = m // (S * N), (m // N) % S, m % N
    ar = torch.arange(ssize, device=patch_feat.device)
    rows = (cy[:, None] + ar)[:, :, None]         # (M, ss, 1)
    cols = (cx[:, None] + ar)[:, None, :]         # (M, 1, ss)
    if isinstance(patch_feat, Upsampled2x):
        # only maps number 0..B-1 of the list are ever indexed (the quirk above): up-sample just those
        idx = [((v // (S * N)) * N + v % N) * S + (v // N) % S for v in range(B)]
        small = patch_feat.materialize(torch.tensor(idx, device=patch_feat.device))        # (B, C, p, p)
        win = small[which[:, None, None], :, rows, cols]                                     # (M, ss, ss, C)
    else:
        win = patch_feat[(mb * N + mn)[:, None, None], ms[:, None, None], :, rows, cols]   # (M, ss, ss, C)
    win = win.permute(0, 3, 1, 2).reshape(B, S, N, C_out, ssize, ssize)[:, 1:].reshape(B * (S - 1) * N, C_out, ssize * ssize)

    sim = torch.einsum("mc,mcr->mr", q, win)
    heat = torch.softmax(sim * (1.0 / C_out ** 0.5), dim=1)                                   # (M', ss*ss)
    lin = torch.linspace(-1.0, 1.0, ssize, device=heat.device, dtype=heat.dtype)
    gx = lin.repeat(ssize)                        # x varies fastest (kornia create_meshgrid, normalized)
    gy = lin.repeat_interleave(ssize)
    grid = torch.stack([gx, gy], -1)              # (ss*ss, 2)
    mean = heat @ grid                            # spatial_expectation2d
    var = heat @ (grid ** 2) - mean ** 2
    std = torch.sqrt(torch.clamp(var, min=1e-10)).sum(-1)
    score = std.reshape(B, S - 1, N)
    return torch.cat([torch.ones_like(score[:, 0:1]), score], dim=1)
