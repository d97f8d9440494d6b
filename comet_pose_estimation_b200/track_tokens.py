"""Fused track-token assembly: what ``BaseTrackerPredictor.forward`` builds every refinement iteration at
comet/models/track_modules/base_track_predictor.py:153-224, as ONE kernel launch:

    x[b,n,s,:] = [ sin/cos(flow) | flow | fcorrs | track_feats | 0 ] + sampled_pos_emb[b,n,:]

``fcorrs`` (the CorrBlock lookup) is computed inside the same kernel and written straight into the token
layout (B,N,S,D) -- no (B,S,N,LW) intermediate, no permute/cat copies, no host-side sincos table."""
from __future__ import annotations

from collections import OrderedDict
from typing import Optional, Union

import torch

from . import _lib
from ._dev import inner_contig, pad_mode, prec_mode, require_cuda, require_no_grad, stream_ptr
from .blocks import CorrBlock, EfficientCorrBlock, Upsampled2x, _make_pyramid, _tc_workspace, _use_tc

lib = _lib.lib


def transformer_dim(corr_levels: int, corr_radius: int, latent_dim: int, fine: bool) -> int:
    """base_track_predictor.py:55-66."""
    d = corr_levels * (corr_radius * 2 + 1) ** 2 + latent_dim * 2
    if fine:
        d += 4 if d % 2 == 0 else 5
    else:
        d += (4 - d % 4) % 4
    return d


# (D, H, W, device) -> channel-last sin/cos table (H, W, D).  The reference rebuilds and uploads the table every
# iteration; here it is kept, LRU-bounded (a tracker uses two shapes: coarse 10.9 MB, fine 0.8 MB).  The building
# stream is synchronised once, so later readers on any stream (or inside a CUDA-graph capture) need no event.
# A batch of several image sizes (track_batch's size groups) uses one coarse table per map size: the bound leaves room
# for 15 sizes besides the fine table, so such batches build no table after their first call.
_TABLES = OrderedDict()
_TABLES_MAX = 16


def _sincos_table_cl(embed_dim: int, H: int, W: int, device) -> torch.Tensor:
    key = (embed_dim, H, W, str(device))
    hit = _TABLES.get(key)
    if hit is None:
        from .utils import get_2d_sincos_pos_embed

        hit = get_2d_sincos_pos_embed(embed_dim, (H, W), device=device)[0].permute(1, 2, 0).contiguous()
        if torch.cuda.is_current_stream_capturing():
            return hit          # built inside a capture: valid for this graph only, not cached
        torch.cuda.current_stream(device).synchronize()
        _TABLES[key] = hit
        while len(_TABLES) > _TABLES_MAX:
            _TABLES.popitem(last=False)
    else:
        _TABLES.move_to_end(key)
    return hit


def sampled_pos_emb(coords0: torch.Tensor, embed_dim: int, H: int, W: int, cached_table: bool = True) -> torch.Tensor:
    """``sample_features4d(get_2d_sincos_pos_embed(D,(H,W)).expand(B,...), coords[:,0])``
    (base_track_predictor.py:200-208) -> (B,N,D); iteration-invariant, so computed once per tracker call.
    The float64-evaluated table depends on (D,H,W) only: it is built once per device (channel-last, so each bilinear tap
    is one contiguous line) and sampled by one kernel.  ``cached_table=False`` evaluates the four taps on the fly
    instead (no table at all; same values)."""
    require_cuda(coords0, "coords0")
    require_no_grad(coords0)
    B, N, two = coords0.shape
    assert two == 2
    c = inner_contig(coords0)
    out = torch.empty((B, N, embed_dim), dtype=torch.float32, device=c.device)
    with torch.cuda.device(c.device):
        if cached_table and B * N:
            tab = _sincos_table_cl(embed_dim, H, W, c.device)
            _lib.check(lib.comet_sample_features4d_cl_f32(tab.data_ptr(), 0, c.data_ptr(), c.stride(0), c.stride(1),
                                                          out.data_ptr(), B, embed_dim, H, W, N, stream_ptr(c.device)))
        else:
            _lib.check(lib.comet_sampled_pos_emb_f32(c.data_ptr(), c.stride(0), c.stride(1), out.data_ptr(), B, N,
                                                     embed_dim, H, W, stream_ptr(c.device)))
    return out


class TrackTokenizer:
    """Per tracker call state of the fused token path: the feature pyramid (built once), the sampled 2-D
    position embedding (built once) and a ``tokens(coords, track_feats)`` method run every iteration."""

    def __init__(self, corr: Union[CorrBlock, EfficientCorrBlock, torch.Tensor, list], coords0: torch.Tensor,
                 tdim: int, num_levels: Optional[int] = None, radius: Optional[int] = None,
                 padding_mode: Optional[str] = None, num_tracks=None, num_frames=None, frame_index=None,
                 group_items=None):
        """``num_tracks`` (B ints or a 1-D tensor): the queries form a padded batch; queries n >= num_tracks[b] are
        padding, their token rows are zeros and cost no correlation work.  ``num_frames`` (likewise): sequence b has the
        first num_frames[b] of the S frames; the token rows of the others are zeros and read nothing.

        ``frame_index`` (B', S) integer tensor: the pyramid holds B_src * S_src source frames (any S_src) and the B'
        items of ``coords0`` read them in their own order -- item i sees source frame ``frame_index[i, s]`` (flat index)
        at position s; any source frame may appear any number of times, in one row or in several.  The items have S
        positions.  The pyramid is prepared once; counts, coordinates and tokens are per item.

        Size groups: ``corr`` a list of G per-group correlation blocks or maps (B_g, S, C, H_g, W_g), maps of different
        sizes.  The items of ``coords0`` are ordered group by group: group g has ``group_items[g]`` items (default
        B_g; required with ``frame_index``, whose rows of group g index group g's source frames).  Each group gets its
        own pyramid and position embedding, and ``tokens`` issues one launch per group into that group's rows of one
        token buffer: the rows are what the call on that group alone computes."""
        self._groups = None
        if isinstance(corr, (list, tuple)):
            from .utils import check_num_tracks

            sizes = [c.shape[0] if isinstance(c, torch.Tensor) else c._pyr.B for c in corr] if group_items is None \
                else list(group_items)
            assert frame_index is None or group_items is not None, "frame_index over size groups needs group_items"
            assert len(sizes) == len(corr) and all(n >= 1 for n in sizes) and sum(sizes) == coords0.shape[0], \
                f"group_items {sizes} do not cover the {coords0.shape[0]} items"
            B = coords0.shape[0]
            counts = None if num_tracks is None else check_num_tracks(num_tracks, B, coords0.shape[1])
            frames = None if num_frames is None else check_num_tracks(num_frames, B, 1 << 30)
            self._groups, at = [], 0
            for c, n in zip(corr, sizes):
                self._groups.append((at, at + n, TrackTokenizer(
                    c, coords0[at:at + n], tdim, num_levels, radius, padding_mode,
                    None if counts is None else counts[at:at + n], None if frames is None else frames[at:at + n],
                    None if frame_index is None else frame_index[at:at + n])))
                at += n
            self.tdim, self.B = tdim, B
            return
        if isinstance(corr, (torch.Tensor, Upsampled2x)):
            assert num_levels is not None and radius is not None
            self.radius = radius
            self.padding_mode = padding_mode or "zeros"
            self._pyr = _make_pyramid(corr, num_levels, radius, self.padding_mode)
        else:
            self._pyr = corr._pyr
            self.radius = corr.radius
            self.padding_mode = padding_mode or ("border" if isinstance(corr, EfficientCorrBlock) else corr.padding_mode)
        assert 0 <= self.radius <= _lib.MAX_RADIUS
        self.tdim = tdim
        p = self._pyr
        self.pos = sampled_pos_emb(coords0, tdim, p.H, p.W)
        self.frame_index = None
        self.B = p.B
        self.S = p.S
        if frame_index is not None:
            assert frame_index.dim() == 2 and frame_index.shape[0] == coords0.shape[0], \
                f"frame_index must be (B', S) with B' = {coords0.shape[0]}, got {tuple(frame_index.shape)}"
            fi = frame_index.to(device=coords0.device, dtype=torch.int32).contiguous()
            assert bool(((fi >= 0) & (fi < p.B * p.S)).all()), f"frame_index outside [0, {p.B * p.S})"
            self.frame_index = fi
            self.B, self.S = coords0.shape[0], int(fi.shape[1])
        self.num_tracks = None
        if num_tracks is not None:
            from .utils import check_num_tracks

            counts = check_num_tracks(num_tracks, coords0.shape[0], coords0.shape[1])
            self.num_tracks = torch.tensor(counts, dtype=torch.int32).to(coords0.device)
        self.num_frames = None
        if num_frames is not None:
            from .utils import check_num_tracks

            frames = check_num_tracks(num_frames, self.B, self.S)
            self.num_frames = torch.tensor(frames, dtype=torch.int32).to(coords0.device)

    def tokens(self, coords: torch.Tensor, track_feats: torch.Tensor, out: Optional[torch.Tensor] = None):
        """coords (B,S,N,2), track_feats (B,S,N,latent) (any outer strides) -> (B,N,S,D_tok) float32."""
        if self._groups is not None:
            B, S, N, _ = coords.shape
            assert B == self.B
            if out is None:
                out = torch.empty((B, N, S, self.tdim), dtype=torch.float32, device=coords.device)
            for r0, r1, tok in self._groups:
                tok.tokens(coords[r0:r1], track_feats[r0:r1], out[r0:r1])
            return out
        p = self._pyr
        B, S, N, D = coords.shape
        assert D == 2
        assert track_feats.shape == (B, S, N, p.C), "track_feats must be (B,S,N,latent) with latent == C"
        assert S == self.S and B == self.B
        require_cuda(coords, "coords")
        require_cuda(track_feats, "track_feats")
        require_no_grad(coords, track_feats)
        c = inner_contig(coords)
        t = inner_contig(track_feats)
        if out is None:
            out = torch.empty((B, N, S, self.tdim), dtype=torch.float32, device=c.device)
        else:
            assert out.shape == (B, N, S, self.tdim) and out.is_contiguous() and out.dtype == torch.float32
        with torch.cuda.device(c.device):
            nt, nf, fi = self.num_tracks, self.num_frames, self.frame_index
            if B * S * N and _use_tc(p, t, self.radius, self.padding_mode):
                head = (p.split.data_ptr(), t.data_ptr(), t.stride(0), t.stride(1), t.stride(2),
                        c.data_ptr(), c.stride(0), c.stride(1), c.stride(2), self.pos.data_ptr(), out.data_ptr())
                tail = (B, S, N, p.C, p.H, p.W, p.num_levels, self.radius, pad_mode(self.padding_mode), prec_mode(),
                        self.tdim, _tc_workspace(p, N, B * S).data_ptr(), stream_ptr(c.device))
                if fi is not None:
                    _lib.check(lib.comet_tc_track_tokens_indexed_f32(
                        *head, None if nt is None else nt.data_ptr(), None if nf is None else nf.data_ptr(), fi.data_ptr(),
                        p.B * p.S, *tail))
                elif nf is not None:
                    _lib.check(lib.comet_tc_track_tokens_varlen_f32(*head, None if nt is None else nt.data_ptr(),
                                                                    nf.data_ptr(), *tail))
                elif nt is None:
                    _lib.check(lib.comet_tc_track_tokens_f32(*head, *tail))
                else:
                    _lib.check(lib.comet_tc_track_tokens_ragged_f32(*head, nt.data_ptr(), *tail))
                return out
            head = (p.fmaps0.data_ptr(), p.pyr.data_ptr(), t.data_ptr(), t.stride(0), t.stride(1), t.stride(2),
                    c.data_ptr(), c.stride(0), c.stride(1), c.stride(2), self.pos.data_ptr(), out.data_ptr())
            tail = (B, S, N, p.C, p.H, p.W, p.num_levels, self.radius, pad_mode(self.padding_mode), prec_mode(),
                    p.layout, self.tdim, stream_ptr(c.device))
            if fi is not None:
                _lib.check(lib.comet_track_tokens_indexed_f32(*head, None if nt is None else nt.data_ptr(),
                                                              None if nf is None else nf.data_ptr(), fi.data_ptr(),
                                                              p.B * p.S, *tail))
            elif nf is not None:
                _lib.check(lib.comet_track_tokens_varlen_f32(*head, None if nt is None else nt.data_ptr(), nf.data_ptr(),
                                                             *tail))
            elif nt is None:
                _lib.check(lib.comet_track_tokens_f32(*head, *tail))
            else:
                _lib.check(lib.comet_track_tokens_ragged_f32(*head, nt.data_ptr(), *tail))
        return out
