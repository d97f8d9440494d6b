"""``CorrBlock`` / ``EfficientCorrBlock`` with the reference's names, signatures and tensor layouts
(comet/models/track_modules/blocks.py:351-484), computed by the fused sm_100a kernels.

Differences a caller can observe: none in results (parity tests) -- but the correlation volume is never
materialised by ``corr()``/``sample()``; ``corrs_pyramid`` is produced lazily only if somebody reads it.  One
consequence: ``corr(targets)`` keeps a *reference* to ``targets`` and the fused kernel reads it at ``sample()`` time,
whereas the reference computes the volume inside ``corr()``.  A caller that mutates ``targets`` in place between the
two calls would get different numbers, so that case is detected (tensor version counter) and refused.  The kernels
are forward-only (the reference runs the tracker under ``torch.no_grad()``)."""
from __future__ import annotations

import ctypes
from typing import List, Optional

import torch

from . import _lib
from ._dev import f32c, inner_contig, pad_mode, prec_mode, require_cuda, require_no_grad, stream_ptr

lib = _lib.lib


def tensor_path_enabled() -> bool:
    """The tcgen05 kernels serve the dense coarse shape; ``_lib.set_option(_lib.OPT_TENSOR_PATH, False)`` forces the
    SIMT kernels (A/B runs)."""
    return bool(lib.comet_has_tensor_path())


class _Pyramid:
    """Level 0 is the caller's tensor; levels 1..L-1 live back to back in one buffer (one allocation,
    written once per tracker call by comet_pyramid_f32)."""

    def __init__(self, fmaps: torch.Tensor, num_levels: int):
        require_cuda(fmaps, "fmaps")
        require_no_grad(fmaps)
        assert fmaps.dim() == 5, "fmaps must be (B, S, C, H, W)"
        B, S, C, H, W = fmaps.shape
        assert 1 <= num_levels <= _lib.MAX_LEVELS, f"num_levels must be in [1, {_lib.MAX_LEVELS}]"
        self.B, self.S, self.C, self.H, self.W = B, S, C, H, W
        self.num_levels = num_levels
        # A dense channels-last view (B,S,C,H,W) with strides (S*H*W*C, H*W*C, 1, W*C, C) -- what a
        # torch.channels_last encoder hands over after a reshape -- is used zero-copy when the fused kernels of the
        # small-map path can read it (one 128-byte line per position); anything else becomes NCHW-contiguous.
        self.cl_input = (fmaps.dtype == torch.float32 and C % 4 == 0 and C <= 64 and B * S > 0 and not fmaps.is_contiguous()
                         and fmaps.permute(0, 1, 3, 4, 2).is_contiguous() and fmaps.data_ptr() % 16 == 0)
        self.fmaps0 = fmaps if self.cl_input else f32c(fmaps)
        n = lib.comet_pyramid_elems(B * S, C, H, W, num_levels)
        assert n >= 0
        self.pyr = torch.empty(max(n, 1), dtype=torch.float32, device=fmaps.device)
        self.split = None  # packed bf16 hi/lo pyramid of the tensor-core path
        self.layout = _lib.PYR_NCHW
        with torch.cuda.device(fmaps.device):
            if B * S > 0 and lib.comet_tc_supported(C, H, W, num_levels, 0, _lib.PAD_ZEROS) and tensor_path_enabled():
                self.split = torch.empty(lib.comet_tc_split_elems(B * S), dtype=torch.bfloat16, device=fmaps.device)
                _lib.check(lib.comet_tc_prepare_f32(self.fmaps0.data_ptr(), self.split.data_ptr(),
                                                    self.pyr.data_ptr(), B * S, C, H, W, num_levels,
                                                    stream_ptr(fmaps.device)))
            elif self.cl_input:
                self.layout = _lib.PYR_ALL_CHANNEL_LAST
                if num_levels > 1:
                    _lib.check(lib.comet_pyramid_cl_f32(self.fmaps0.data_ptr(), self.pyr.data_ptr(), B * S, C, H, W,
                                                        num_levels, _lib.FMAPS_CHANNEL_LAST, stream_ptr(fmaps.device)))
            elif W <= 32 and H <= 33 and C % 4 == 0 and C <= 64 and num_levels > 1:
                # small maps (fine tracker patches): levels >= 1 channel-last, one contiguous line per position
                self.layout = _lib.PYR_CHANNEL_LAST
                _lib.check(lib.comet_pyramid_cl_f32(self.fmaps0.data_ptr(), self.pyr.data_ptr(), B * S, C, H, W,
                                                    num_levels, _lib.FMAPS_NCHW, stream_ptr(fmaps.device)))
            else:
                _lib.check(lib.comet_pyramid_f32(self.fmaps0.data_ptr(), self.pyr.data_ptr(), B * S, C, H, W,
                                                 num_levels, stream_ptr(fmaps.device)))
        self.levels: List[torch.Tensor] = [fmaps]
        self._ws = {}  # scratch of the tensor path (sorted query order + job list) per CUDA stream
        h, w = H, W
        for l in range(1, num_levels):
            h, w = h // 2, w // 2
            off = lib.comet_pyramid_offset(B * S, C, H, W, l)
            flat = self.pyr[off: off + B * S * C * h * w]
            if self.layout != _lib.PYR_NCHW:
                self.levels.append(flat.view(B, S, h, w, C).permute(0, 1, 4, 2, 3))  # same values, strided view
            else:
                self.levels.append(flat.view(B, S, C, h, w))


class Upsampled2x:
    """A (B, S, C, 2Hs-1, 2Ws-1) feature tensor that is *defined* as
    ``F.interpolate(src, (2Hs-1, 2Ws-1), mode="bilinear", align_corners=True)`` of a half-resolution map ``src``
    (B, S, C, Hs, Ws) but never materialised: what ``ShallowEncoder`` computes right before its last resize
    (blocks.py:176-190).  ``CorrBlock`` / ``BaseTrackerPredictor`` of this package accept it in place of ``fmaps`` and
    evaluate pyramid levels 0 and 1 from ``src`` inside the fused lookup (COMET_PYR_UP2_SOURCE, csrc/corr_lookup_up2.cu):
    the 1 GB-per-sequence up-sampled tensor of the fine tracker is neither written nor read.  ``materialize()`` gives
    the ordinary tensor (any subset of maps) for callers that need values, e.g. ``compute_score_fn``."""

    def __init__(self, src: torch.Tensor):
        require_cuda(src, "src")
        require_no_grad(src)
        assert src.dim() == 5, "src must be (B, S, C, Hs, Ws)"
        B, S, C, Hs, Ws = src.shape
        src = src if src.dtype == torch.float32 else src.float()
        if not (src.permute(0, 1, 3, 4, 2).is_contiguous() and src.data_ptr() % 16 == 0):
            src = src.permute(0, 1, 3, 4, 2).contiguous().permute(0, 1, 4, 2, 3)   # channels-last memory, same shape
        self.src = src
        self.shape = torch.Size((B, S, C, 2 * Hs - 1, 2 * Ws - 1))
        self.device, self.dtype = src.device, torch.float32

    def dim(self) -> int:
        return 5

    def materialize(self, index=None) -> torch.Tensor:
        """The up-sampled tensor itself, (B,S,C,H,W), or maps ``index`` of its (B*S) flattening -> (len, C, H, W)."""
        from .utils import upsample_bilinear_align_corners

        B, S, C, H, W = self.shape
        flat = self.src.permute(0, 1, 3, 4, 2).reshape(B * S, self.src.shape[3], self.src.shape[4], C).permute(0, 3, 1, 2)
        if index is not None:
            return upsample_bilinear_align_corners(flat[index].contiguous(memory_format=torch.channels_last), (H, W))
        return upsample_bilinear_align_corners(flat, (H, W)).permute(0, 2, 3, 1).reshape(B, S, H, W, C).permute(0, 1, 4, 2, 3)


class _PyramidUp2:
    """Pyramid state of the COMET_PYR_UP2_SOURCE layout: the source map (level 0 and 1 are stencils of it) and the
    pooled level 2; duck-types ``_Pyramid`` for the fused lookup / token entry points."""

    def __init__(self, up: Upsampled2x, num_levels: int):
        B, S, C, H, W = up.shape
        self.B, self.S, self.C, self.H, self.W = B, S, C, H, W
        self.num_levels = num_levels
        self.up = up
        self.fmaps0 = up.src                      # passed as `fmaps`: the half-resolution source
        self.cl_input = True
        self.split = None
        self.layout = _lib.PYR_UP2_SOURCE
        self._ws = {}
        Hs, Ws = up.src.shape[-2:]
        n = lib.comet_pyramid_up2_elems(B * S, C, Hs, Ws)
        assert n >= 0
        self.pyr = torch.empty(max(n, 1), dtype=torch.float32, device=up.device)   # level 2 only, channel-last
        with torch.cuda.device(up.device):
            if B * S:
                _lib.check(lib.comet_pyramid_up2_f32(up.src.data_ptr(), self.pyr.data_ptr(), B * S, C, Hs, Ws,
                                                     stream_ptr(up.device)))
        self._levels = None

    @property
    def levels(self) -> List[torch.Tensor]:
        """``fmaps_pyramid`` as the reference stores it (values only needed by callers that read the attribute)."""
        if self._levels is None:
            self._levels = _Pyramid(self.up.materialize(), self.num_levels).levels
        return self._levels


def up2_supported(fmaps, num_levels: int, radius: int, padding_mode: str) -> bool:
    if not isinstance(fmaps, Upsampled2x):
        return False
    B, S, C, H, W = fmaps.shape
    with torch.cuda.device(fmaps.device):
        return bool(lib.comet_up2_supported(C, H, W, num_levels, radius, pad_mode(padding_mode)))


def _make_pyramid(fmaps, num_levels: int, radius: int, padding_mode: str):
    if isinstance(fmaps, Upsampled2x):
        if up2_supported(fmaps, num_levels, radius, padding_mode):
            return _PyramidUp2(fmaps, num_levels)
        fmaps = fmaps.materialize()    # shape the specialised kernel does not serve: the ordinary path
    return _Pyramid(fmaps, num_levels)


def _tc_workspace(pyr: "_Pyramid", N: int, BS: Optional[int] = None) -> torch.Tensor:
    """Scratch of the tensor path, one buffer per CUDA stream (two streams driving the same CorrBlock never share a
    plan).  It grows only when a larger N arrives: under CUDA-graph capture call once with the largest N first.  ``BS``:
    the (item, position) frames of the call when they differ from the pyramid's (a frame table)."""
    need = lib.comet_tc_workspace_bytes(pyr.B * pyr.S if BS is None else BS, N)
    key = stream_ptr(pyr.fmaps0.device)
    ws = pyr._ws.get(key)
    if ws is None or ws.numel() * 4 < need:
        ws = torch.empty((need + 3) // 4, dtype=torch.int32, device=pyr.fmaps0.device)
        pyr._ws[key] = ws
    return ws


def _use_tc(pyr: "_Pyramid", t: torch.Tensor, radius: int, padding: str, level_stride: int = 0) -> bool:
    return (pyr.split is not None and level_stride == 0 and padding == "zeros" and radius <= 4
            and t.data_ptr() % 16 == 0 and all(st % 4 == 0 for st in t.stride()[:3]))


def _fused_lookup(pyr: _Pyramid, targets, coords, radius, padding, level_stride=0):
    B, S, N, D = coords.shape
    assert D == 2
    require_cuda(coords, "coords")
    require_cuda(targets, "targets")
    require_no_grad(coords, targets)
    t = inner_contig(targets)
    c = inner_contig(coords)
    Wr = 2 * radius + 1
    out = torch.empty((B, S, N, pyr.num_levels * Wr * Wr), dtype=torch.float32, device=coords.device)
    with torch.cuda.device(coords.device):
        if B * S * N and _use_tc(pyr, t, radius, padding, level_stride):
            _lib.check(lib.comet_tc_corr_lookup_f32(
                pyr.split.data_ptr(), t.data_ptr(), t.stride(0), t.stride(1), t.stride(2),
                c.data_ptr(), c.stride(0), c.stride(1), c.stride(2),
                out.data_ptr(), out.stride(0), out.stride(1), out.stride(2),
                B, S, N, pyr.C, pyr.H, pyr.W, pyr.num_levels, radius, pad_mode(padding), prec_mode(),
                _tc_workspace(pyr, N).data_ptr(), stream_ptr(coords.device)))
            return out
        _lib.check(lib.comet_corr_lookup_f32(
            pyr.fmaps0.data_ptr(), pyr.pyr.data_ptr(),
            t.data_ptr(), t.stride(0), t.stride(1), t.stride(2), level_stride,
            c.data_ptr(), c.stride(0), c.stride(1), c.stride(2),
            out.data_ptr(), out.stride(0), out.stride(1), out.stride(2),
            B, S, N, pyr.C, pyr.H, pyr.W, pyr.num_levels, radius, pad_mode(padding), prec_mode(), pyr.layout,
            stream_ptr(coords.device)))
    return out


class CorrBlock:
    """Drop-in for blocks.py:351-429.  Plain class (not an nn.Module), no parameters, stateful between
    ``corr()`` and ``sample()``."""

    def __init__(self, fmaps, num_levels=4, radius=4, multiple_track_feats=False, padding_mode="zeros"):
        B, S, C, H, W = fmaps.shape
        self.S, self.C, self.H, self.W = S, C, H, W
        self.padding_mode = padding_mode
        self.num_levels = num_levels
        self.radius = radius
        self.multiple_track_feats = multiple_track_feats
        pad_mode(padding_mode)  # validate early
        assert 0 <= radius <= _lib.MAX_RADIUS, f"radius must be in [0, {_lib.MAX_RADIUS}]"
        if multiple_track_feats and isinstance(fmaps, Upsampled2x):
            fmaps = fmaps.materialize()     # per-level targets are served by the general kernel only
        self._pyr = _make_pyramid(fmaps, num_levels, radius, padding_mode)
        self._targets: Optional[torch.Tensor] = None
        self._volumes: Optional[List[torch.Tensor]] = None

    @classmethod
    def from_upsampled(cls, src, num_levels=4, radius=4, multiple_track_feats=False, padding_mode="zeros"):
        """``CorrBlock(F.interpolate(src, (2Hs-1, 2Ws-1), bilinear, align_corners=True), ...)`` without the up-sampled
        tensor: ``src`` (B,S,C,Hs,Ws) is the patch encoder's half-resolution output (see :class:`Upsampled2x`)."""
        return cls(src if isinstance(src, Upsampled2x) else Upsampled2x(src), num_levels, radius, multiple_track_feats,
                   padding_mode)

    @property
    def fmaps_pyramid(self):
        return self._pyr.levels

    def corr(self, targets):
        B, S, N, C = targets.shape
        if self.multiple_track_feats:
            C = C // self.num_levels
        assert C == self.C
        assert S == self.S
        require_cuda(targets, "targets")
        self._targets = targets
        self._targets_version = targets._version
        self._volumes = None

    def _check_targets_unchanged(self):
        if self._targets._version != self._targets_version:
            raise RuntimeError(
                "CorrBlock: `targets` was modified in place after corr(). The reference computes the correlation "
                "volume inside corr(); this implementation reads `targets` when sample() / corrs_pyramid is "
                "evaluated. Call corr() again with the updated tensor.")

    @property
    def corrs_pyramid(self):
        """List of (B,S,N,H_l,W_l) volumes, as the reference stores after ``corr()`` (blocks.py:420-429).
        Materialised on first access only; ``sample()`` does not need it."""
        if self._targets is None:
            raise AttributeError("'CorrBlock' object has no attribute 'corrs_pyramid' (call corr() first)")
        if self._volumes is None:
            self._check_targets_unchanged()
            p = self._pyr
            if isinstance(p, _PyramidUp2):   # API completeness only: volumes of the materialised pyramid
                p = _Pyramid(p.up.materialize(), p.num_levels)
            B, S, N, _ = self._targets.shape
            t = f32c(self._targets).view(B * S, N, -1)
            vols = []
            mode = prec_mode()
            with torch.cuda.device(t.device):
                if B * S * N and not self.multiple_track_feats and _use_tc(p, t.view(B, S, N, -1), 0, "zeros"):
                    for f in p.levels:
                        vols.append(torch.empty((B, S, N) + tuple(f.shape[-2:]), dtype=torch.float32,
                                                device=t.device))
                    ptrs = (ctypes.c_void_p * len(vols))(*[v.data_ptr() for v in vols])
                    t4 = t.view(B, S, N, -1)
                    _lib.check(lib.comet_tc_corr_volume_f32(
                        p.split.data_ptr(), t4.data_ptr(), t4.stride(0), t4.stride(1), t4.stride(2), ptrs,
                        B, S, N, p.C, p.H, p.W, p.num_levels, mode, _tc_workspace(p, N).data_ptr(),
                        stream_ptr(t.device)))
                    if mode == _lib.PREC_BF16_AUTOCAST:
                        vols = [v.to(torch.bfloat16) for v in vols]
                    self._volumes = vols
                    return self._volumes
                for l, f in enumerate(p.levels):
                    h, w = f.shape[-2:]
                    tl = t[..., l * self.C:(l + 1) * self.C] if self.multiple_track_feats else t
                    fl = p.fmaps0 if (l == 0 and not p.cl_input) else f.contiguous()
                    v = torch.empty((B, S, N, h, w), dtype=torch.float32, device=t.device)
                    for b0 in range(0, B * S, 32768):  # gridDim.z limit
                        nb = min(32768, B * S - b0)
                        _lib.check(lib.comet_corr_volume_f32(
                            tl[b0:].data_ptr(), tl.stride(0), tl.stride(1),
                            fl.reshape(B * S, self.C, h * w)[b0:].data_ptr(),
                            v.view(B * S, N, h * w)[b0:].data_ptr(), nb, N, self.C, h * w, mode,
                            stream_ptr(t.device)))
                    vols.append(v.to(torch.bfloat16) if mode == _lib.PREC_BF16_AUTOCAST else v)
            self._volumes = vols
        return self._volumes

    def sample(self, coords):
        B, S, N, D = coords.shape
        assert D == 2
        if self._targets is None:
            raise AttributeError("'CorrBlock' object has no attribute 'corrs_pyramid' (call corr() first)")
        self._check_targets_unchanged()
        return _fused_lookup(self._pyr, self._targets, coords, self.radius, self.padding_mode,
                             self.C if self.multiple_track_feats else 0)


class EfficientCorrBlock:
    """Drop-in for blocks.py:432-484: same pyramid, ``sample(coords, target)`` with *border* padding."""

    def __init__(self, fmaps, num_levels=4, radius=4):
        self.num_levels = num_levels
        self.radius = radius
        assert 0 <= radius <= _lib.MAX_RADIUS, f"radius must be in [0, {_lib.MAX_RADIUS}]"
        self._pyr = _make_pyramid(fmaps, num_levels, radius, "border")
        self.fmaps_pyramid = self._pyr.levels

    def sample(self, coords, target):
        B, S, N, D = coords.shape
        assert D == 2
        assert target.shape[-1] == self._pyr.C and target.shape[1] == self._pyr.S
        return _fused_lookup(self._pyr, target, coords, self.radius, "border")
