"""Track-update transformer used between hot-path iterations (SURVEY.md 8f, rank 1).

``EfficientUpdateFormer`` owns the parameters under the reference's names (comet/models/track_modules/blocks.py:205-348,
attention blocks comet/models/modules.py:248-344), so reference checkpoints (``track_predictor.*.updateformer.*`` keys)
load unchanged.  CUDA inference runs on this package's own sm_100a kernels (:mod:`.update_former_tc`: tcgen05 GEMMs
with fused bias / GELU / residual epilogues, LayerNorm and attention kernels); the plain ``torch.nn`` forward below is
the definition those kernels are tested against, and what runs on CPU tensors (host-logic tests), under autograd, and
for shapes the kernels do not serve (head_dim not a multiple of 4).

Quirks preserved (they change numerics): both block types add the attention output to the *normalised* input
(``x = norm1(x); x = x + attn(x)``), the virtual-track parameter is spelled ``virual_tracks``, and the initial
projected tokens are added back before the flow head.
"""
from __future__ import annotations

import torch
import torch.nn as nn

# False keeps CUDA inference on the torch.nn forward as well (A/B timing in bench.py, parity tests)
USE_TC_KERNELS = True


class _FeedForward(nn.Module):
    """fc1 -> GELU -> fc2 (parameter names of the reference's ``Mlp``, modules.py:119-154)."""

    def __init__(self, dim: int, hidden: int):
        super().__init__()
        self.fc1 = nn.Linear(dim, hidden)
        self.act = nn.GELU()
        self.fc2 = nn.Linear(hidden, dim)

    def forward(self, x):
        return self.fc2(self.act(self.fc1(x)))


class SelfAttnBlock(nn.Module):
    """Reference ``AttnBlock`` (modules.py:248-297)."""

    def __init__(self, dim: int, heads: int, mlp_ratio: float = 4.0):
        super().__init__()
        self.norm1 = nn.LayerNorm(dim, elementwise_affine=False, eps=1e-6)
        self.norm2 = nn.LayerNorm(dim, elementwise_affine=False, eps=1e-6)
        self.attn = nn.MultiheadAttention(embed_dim=dim, num_heads=heads, batch_first=True)
        self.mlp = _FeedForward(dim, int(dim * mlp_ratio))

    def forward(self, x, mask=None):
        x = self.norm1(x)
        x = x + self.attn(x, x, x)[0]  # same call as the reference (weights path), keeps the arithmetic identical
        return x + self.mlp(self.norm2(x))


class CrossAttnBlock(nn.Module):
    """Reference ``CrossAttnBlock`` (modules.py:300-344)."""

    def __init__(self, dim: int, context_dim: int, heads: int = 1, mlp_ratio: float = 4.0):
        super().__init__()
        self.norm1 = nn.LayerNorm(dim, elementwise_affine=False, eps=1e-6)
        self.norm_context = nn.LayerNorm(dim)
        self.norm2 = nn.LayerNorm(dim, elementwise_affine=False, eps=1e-6)
        self.cross_attn = nn.MultiheadAttention(embed_dim=dim, num_heads=heads, batch_first=True)
        self.mlp = _FeedForward(dim, int(dim * mlp_ratio))

    def forward(self, x, context, mask=None):
        x = self.norm1(x)
        context = self.norm_context(context)
        x = x + self.cross_attn(x, context, context, attn_mask=mask)[0]
        return x + self.mlp(self.norm2(x))


class EfficientUpdateFormer(nn.Module):
    """(B, N, T, input_dim) tokens -> (B, N, T, output_dim) updates: alternating attention over time (per track)
    and over space (tracks <-> 64 learned virtual tracks)."""

    def __init__(self, space_depth=6, time_depth=6, input_dim=320, hidden_size=384, num_heads=8, output_dim=130,
                 mlp_ratio=4.0, add_space_attn=True, num_virtual_tracks=64):
        super().__init__()
        self.out_channels = 2
        self.num_heads = num_heads
        self.hidden_size = hidden_size
        self.add_space_attn = add_space_attn
        self.num_virtual_tracks = num_virtual_tracks
        self.input_transform = nn.Linear(input_dim, hidden_size, bias=True)
        self.flow_head = nn.Linear(hidden_size, output_dim, bias=True)
        self.virual_tracks = (nn.Parameter(torch.randn(1, num_virtual_tracks, 1, hidden_size))
                              if add_space_attn else None)
        self.time_blocks = nn.ModuleList(SelfAttnBlock(hidden_size, num_heads, mlp_ratio) for _ in range(time_depth))
        if add_space_attn:
            self.space_virtual_blocks = nn.ModuleList(
                SelfAttnBlock(hidden_size, num_heads, mlp_ratio) for _ in range(space_depth))
            self.space_point2virtual_blocks = nn.ModuleList(
                CrossAttnBlock(hidden_size, hidden_size, num_heads, mlp_ratio) for _ in range(space_depth))
            self.space_virtual2point_blocks = nn.ModuleList(
                CrossAttnBlock(hidden_size, hidden_size, num_heads, mlp_ratio) for _ in range(space_depth))
            assert len(self.time_blocks) >= len(self.space_virtual2point_blocks)

    def forward(self, input_tensor, mask=None, num_tracks=None, num_frames=None):
        """``num_tracks`` (B ints or a 1-D tensor): ``input_tensor`` is a padded batch (B, N_max, T, input_dim) of sequences
        with ``num_tracks[b]`` tracks each.  ``num_frames`` (likewise): sequence b has ``num_frames[b]`` of the T frames.
        Sequence b's rows get what the forward of ``input_tensor[b:b+1, :num_tracks[b], :num_frames[b]]`` alone returns;
        rows past its counts are zeros."""
        ragged = num_tracks is not None or num_frames is not None
        if ragged:
            assert mask is None, "num_tracks / num_frames and mask cannot be combined"
            from .utils import check_num_tracks

            B, N, T = input_tensor.shape[:3]
            counts = None if num_tracks is None else check_num_tracks(num_tracks, B, N)
            frames = None if num_frames is None else check_num_tracks(num_frames, B, T)
        if (USE_TC_KERNELS and mask is None and input_tensor.is_cuda and not torch.is_grad_enabled()):
            from . import update_former_tc as tc

            if tc.supported(self, input_tensor) and (not ragged or tc.ragged_supported(self)):
                autocast = torch.is_autocast_enabled("cuda") and torch.get_autocast_dtype("cuda") == torch.bfloat16
                if ragged:
                    dev = input_tensor.device
                    dev_counts = None if counts is None else torch.tensor(counts, dtype=torch.int32).to(dev, non_blocking=True)
                    dev_frames = None if frames is None else torch.tensor(frames, dtype=torch.int32).to(dev, non_blocking=True)
                    if dev_frames is None:
                        return tc.forward_ragged(self, input_tensor.float(), 1 if autocast else 3, dev_counts)
                    return tc.forward_ragged(self, input_tensor.float(), 1 if autocast else 3, dev_counts, dev_frames)
                return tc.forward(self, input_tensor.float(), 1 if autocast else 3)
        if ragged:
            return self._forward_ragged_torch(input_tensor, counts, frames)
        return self._forward_torch(input_tensor, mask)

    def _forward_ragged_torch(self, input_tensor, counts, frames=None):
        """The per-sequence definition of the ragged forward: each sequence alone, re-padded with zeros."""
        B, N, T = input_tensor.shape[:3]
        counts = [N] * B if counts is None else counts
        frames = [T] * B if frames is None else frames
        outs = [self._forward_torch(input_tensor[b:b + 1, :n, :s]) for b, (n, s) in enumerate(zip(counts, frames))]
        out = outs[0].new_zeros((B, N, T) + tuple(outs[0].shape[3:]))
        for b, (o, n, s) in enumerate(zip(outs, counts, frames)):
            out[b, :n, :s] = o[0]
        return out

    def _forward_torch(self, input_tensor, mask=None):
        tokens = self.input_transform(input_tensor)
        skip = tokens
        B, _, T, _ = tokens.shape
        V = self.num_virtual_tracks
        if self.add_space_attn:
            tokens = torch.cat([tokens, self.virual_tracks.repeat(B, 1, T, 1)], dim=1)
        N = tokens.shape[1]
        every = len(self.time_blocks) // len(self.space_virtual_blocks) if self.add_space_attn else 0
        j = 0
        for i, time_block in enumerate(self.time_blocks):
            tokens = time_block(tokens.contiguous().view(B * N, T, -1)).view(B, N, T, -1)
            if self.add_space_attn and i % every == 0:
                st = tokens.permute(0, 2, 1, 3).contiguous().view(B * T, N, -1)
                points, virt = st[:, : N - V], st[:, N - V:]
                virt = self.space_virtual2point_blocks[j](virt, points, mask=mask)
                virt = self.space_virtual_blocks[j](virt)
                points = self.space_point2virtual_blocks[j](points, virt, mask=mask)
                tokens = torch.cat([points, virt], dim=1).view(B, T, N, -1).permute(0, 2, 1, 3)
                j += 1
        if self.add_space_attn:
            tokens = tokens[:, : N - V]
        return self.flow_head(tokens + skip)
