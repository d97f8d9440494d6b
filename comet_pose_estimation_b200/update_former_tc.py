"""sm_100a execution of ``EfficientUpdateFormer`` (comet/models/track_modules/blocks.py:205-348) and its
``AttnBlock`` / ``CrossAttnBlock`` / ``Mlp`` (comet/models/modules.py:119-154, :248-344): every Linear runs on the tcgen05
GEMM of ``csrc/gemm_tc.cu`` with bias / GELU / residual fused into its epilogue, LayerNorm and the short-sequence
attention run in ``csrc/transformer.cu``.  ``update_former.EfficientUpdateFormer`` owns the parameters (reference
state-dict keys) and calls :func:`forward` for CUDA inference.

Data flow.  Token rows keep ONE order for the whole transformer -- (track n, frame t), points first, the 64 virtual
tracks after them -- and the attention kernel takes batch / position strides, so neither of the reference's
rearrangements ("(b n) t c" for time attention, "(b t) n c" for space attention, blocks.py:312-338) nor its
``torch.cat`` copies exist.  Activations that feed a GEMM are written by their producer directly as bf16 planes (see
include/comet_b200.h): ``np = 3`` planes give float32-grade products (six tensor-core passes), ``np = 1`` is what
``torch.autocast(bf16)`` makes of the reference's Linear layers (COMET ships ``mixed_precision: bf16``).

Quirks preserved (they change numerics): both block types add the attention output to the *normalised* input
(``x = norm1(x); x = x + attn(x)``), and the projected input tokens are added back before the flow head.
"""
from __future__ import annotations

from typing import Dict, Tuple

import torch

from . import _lib
from ._dev import stream_ptr

lib = _lib.lib


def supported(m, x: torch.Tensor) -> bool:
    """Shapes the kernels serve: head_dim a multiple of 4 and <= 64, hidden <= 1024, float32 CUDA tokens."""
    if not (isinstance(x, torch.Tensor) and x.is_cuda and x.dtype == torch.float32 and x.dim() == 4):
        return False
    D, H = m.hidden_size, m.num_heads
    if D % H or (D // H) % 4 or D // H > 64 or D > 1024 or D % 8:
        return False
    with torch.cuda.device(x.device):
        return bool(lib.comet_has_tensor_path() or _device_ok())


def _device_ok() -> bool:
    return torch.cuda.get_device_capability()[0] == 10


def _ceil8(k: int) -> int:
    return (k + 7) // 8 * 8


def _to_planes(w: torch.Tensor, np_: int) -> torch.Tensor:
    """(N, K) float32 -> (np, N, ceil8(K)) bf16 planes (zero padded along K)."""
    N, K = w.shape
    out = torch.zeros((np_, N, _ceil8(K)), dtype=torch.bfloat16, device=w.device)
    r = w.float()
    for i in range(np_):
        b = r.to(torch.bfloat16)
        out[i, :, :K] = b
        r = r - b.float()
    return out


class _Weights:
    """bf16 planes of every Linear weight of one module, rebuilt when a parameter changes (load_state_dict, .to())."""

    def __init__(self):
        self.cache: Dict[Tuple[int, int], Tuple[tuple, torch.Tensor]] = {}

    def planes(self, w: torch.Tensor, np_: int) -> torch.Tensor:
        key = (id(w), np_)
        tag = (w.data_ptr(), w._version, tuple(w.shape), str(w.device))
        hit = self.cache.get(key)
        if hit is None or hit[0] != tag:
            hit = (tag, _to_planes(w.detach(), np_))
            self.cache[key] = hit
        return hit[1]


class _Run:
    """One forward: thin wrappers around the C entry points operating on row-major float32 matrices and plane tensors."""

    def __init__(self, weights: _Weights, np_: int, device):
        self.w, self.np, self.dev = weights, np_, device
        self.stream = stream_ptr(device)

    def new_f32(self, rows: int, cols: int) -> torch.Tensor:
        return torch.empty((rows, cols), dtype=torch.float32, device=self.dev)

    def new_planes(self, rows: int, cols: int) -> torch.Tensor:
        return torch.empty((self.np, rows, _ceil8(cols)), dtype=torch.bfloat16, device=self.dev)

    def split(self, x: torch.Tensor) -> torch.Tensor:
        rows, cols = x.shape
        p = self.new_planes(rows, cols)
        if p.shape[2] != cols:
            p.zero_()
        _lib.check(lib.comet_split_planes_f32(x.data_ptr(), x.stride(0), p.data_ptr(), p.stride(0), p.stride(1), rows,
                                              cols, self.np, self.stream))
        return p

    def layernorm(self, x: torch.Tensor, norm: torch.nn.LayerNorm, want_f32: bool, want_planes: bool = True):
        rows, D = x.shape
        out = self.new_f32(rows, D) if want_f32 else None
        p = self.new_planes(rows, D) if want_planes else None
        g = norm.weight.data_ptr() if norm.elementwise_affine else None
        b = norm.bias.data_ptr() if norm.elementwise_affine else None
        _lib.check(lib.comet_layernorm_planes_f32(
            x.data_ptr(), x.stride(0), g, b, float(norm.eps), out.data_ptr() if want_f32 else None, D,
            p.data_ptr() if want_planes else None, p.stride(0) if want_planes else 0, p.stride(1) if want_planes else 0,
            self.np if want_planes else 0, rows, D, self.stream))
        return out, p

    def linear(self, xp: torch.Tensor, weight: torch.Tensor, bias, n0: int = 0, n1: int = None, resid=None, out=None,
               want_f32: bool = True, want_planes: bool = False, gelu: bool = False):
        """rows [n0, n1) of ``weight`` (N_total, K) applied to planes ``xp`` (np, M, Kp)."""
        wp = self.w.planes(weight, self.np)
        n1 = weight.shape[0] if n1 is None else n1
        N, K = n1 - n0, weight.shape[1]
        M = xp.shape[1]
        assert xp.shape[2] == wp.shape[2], "operand planes disagree on the padded K"
        if want_f32 and out is None:
            out = self.new_f32(M, N)
        op = self.new_planes(M, N) if want_planes else None
        wsub = wp[:, n0:n1]
        _lib.check(lib.comet_linear_tc(
            xp.data_ptr(), xp.stride(0), xp.stride(1), wsub.data_ptr(), wp.stride(0), wp.stride(1), self.np,
            bias[n0:n1].data_ptr() if bias is not None else None,
            resid.data_ptr() if resid is not None else None, resid.stride(0) if resid is not None else 0,
            out.data_ptr() if want_f32 else None, out.stride(0) if want_f32 else 0,
            op.data_ptr() if want_planes else None, op.stride(0) if want_planes else 0, op.stride(1) if want_planes else 0,
            self.np if want_planes else 0, int(gelu), M, N, K, self.stream))
        return out, op

    def attention(self, q, k, v, B: int, H: int, Lq: int, Lk: int, dh: int, q_sb, q_si, k_sb, k_si, rows_out: int, D: int,
                  o_sb, o_si):
        """q / k / v: float32 views (column slices of GEMM outputs) whose rows are tokens; strides in elements."""
        op = self.new_planes(rows_out, D)
        _lib.check(lib.comet_attention_planes_f32(q.data_ptr(), q_sb, q_si, k.data_ptr(), k_sb, k_si, v.data_ptr(), k_sb, k_si,
                                                  op.data_ptr(), op.stride(0), o_sb, o_si, self.np, B, H, Lq, Lk, dh,
                                                  self.stream))
        return op

    def attention_varlen(self, q, k, v, H: int, dh: int, step: int, items, q_off, q_len, k_off, k_len, lq, lk, group,
                         rows_out: int, D: int, zero: bool = False):
        """Every item of ``items`` in one call: item i's position j is row ``q_off[i] + j * step`` of q / of the output
        and row ``k_off[i] + j * step`` of k / v (int32 device arrays); ``lq`` / ``lk`` bound the lengths (0 skips an
        item).  ``group``: the problem count that selects each item's kernel family, an int or ``(groups, lo, hi)`` with
        ``groups`` an int32 device array of per-item counts in [lo, hi].  ``zero``: the output rows no item writes
        (padded queries) are zeros instead of unset."""
        op = self.new_planes(rows_out, D)
        if zero:
            op.zero_()
        assert k.stride(0) == v.stride(0)
        groups, glo, ghi = (None, group, group) if isinstance(group, int) else group
        _lib.check(lib.comet_attention_varlen_grouped_planes_f32(
            q.data_ptr(), q.stride(0), step, k.data_ptr(), k.stride(0), step, v.data_ptr(), op.data_ptr(), op.stride(0),
            op.stride(1), self.np, items, H, dh, q_off.data_ptr(), q_len.data_ptr(), k_off.data_ptr(), k_len.data_ptr(),
            lq[0], lq[1], lk[0], lk[1], None if groups is None else groups.data_ptr(), glo, ghi, self.stream))
        return op

    def mlp_tail(self, y: torch.Tensor, blk, out: torch.Tensor):
        """out = y + fc2(GELU(fc1(norm2(y))))   (modules.py:119-154; norm2 without affine)."""
        _, ynp = self.layernorm(y, blk.norm2, want_f32=False)
        _, hp = self.linear(ynp, blk.mlp.fc1.weight, blk.mlp.fc1.bias, want_f32=False, want_planes=True, gelu=True)
        self.linear(hp, blk.mlp.fc2.weight, blk.mlp.fc2.bias, resid=y, out=out)

    def self_block(self, x: torch.Tensor, blk, nbatch: int, L: int, sb: int, si: int, H: int):
        """Reference ``AttnBlock`` in place on the rows of ``x`` (rows, D): ``nbatch`` sequences of ``L`` positions whose
        rows are ``b * sb + i * si`` (in rows)."""
        rows, D = x.shape
        dh = D // H
        xn, xnp = self.layernorm(x, blk.norm1, want_f32=True)
        qkv, _ = self.linear(xnp, blk.attn.in_proj_weight, blk.attn.in_proj_bias)
        ld = qkv.stride(0)
        ctx = self.attention(qkv[:, :D], qkv[:, D:2 * D], qkv[:, 2 * D:], nbatch, H, L, L, dh, sb * ld, si * ld, sb * ld, si * ld,
                             rows, D, sb * _ceil8(D), si * _ceil8(D))
        y, _ = self.linear(ctx, blk.attn.out_proj.weight, blk.attn.out_proj.bias, resid=xn)
        self.mlp_tail(y, blk, out=x)

    def cross_block(self, x: torch.Tensor, ctxt: torch.Tensor, blk, T: int, H: int):
        """Reference ``CrossAttnBlock`` in place on ``x`` (nx*T, D) attending to ``ctxt`` (nc*T, D); rows are (track, frame):
        one attention problem per frame over the tracks."""
        rows, D = x.shape
        dh = D // H
        nx, nc = rows // T, ctxt.shape[0] // T
        xn, xnp = self.layernorm(x, blk.norm1, want_f32=True)
        _, cnp = self.layernorm(ctxt, blk.norm_context, want_f32=False)
        a = blk.cross_attn
        q, _ = self.linear(xnp, a.in_proj_weight, a.in_proj_bias, 0, D)
        kv, _ = self.linear(cnp, a.in_proj_weight, a.in_proj_bias, D, 3 * D)
        ctx = self.attention(q, kv[:, :D], kv[:, D:], T, H, nx, nc, dh, q.stride(0), T * q.stride(0), kv.stride(0),
                             T * kv.stride(0), rows, D, _ceil8(D), T * _ceil8(D))
        y, _ = self.linear(ctx, a.out_proj.weight, a.out_proj.bias, resid=xn)
        self.mlp_tail(y, blk, out=x)


    def self_block_varlen(self, x: torch.Tensor, blk, H: int, step: int, items: int, off, length, lrange, group):
        """``self_block`` over ``items`` sequences of rows at once: item i has ``length[i]`` positions at rows
        ``off[i] + j * step`` (the virtual tracks of every (sequence, frame), or the frames of every track)."""
        rows, D = x.shape
        xn, xnp = self.layernorm(x, blk.norm1, want_f32=True)
        qkv, _ = self.linear(xnp, blk.attn.in_proj_weight, blk.attn.in_proj_bias)
        ctx = self.attention_varlen(qkv[:, :D], qkv[:, D:2 * D], qkv[:, 2 * D:], H, D // H, step, items, off, length, off,
                                    length, lrange, lrange, group, rows, D, zero=lrange[0] != lrange[1])
        y, _ = self.linear(ctx, blk.attn.out_proj.weight, blk.attn.out_proj.bias, resid=xn)
        self.mlp_tail(y, blk, out=x)

    def cross_block_varlen(self, x: torch.Tensor, ctxt: torch.Tensor, blk, H: int, step: int, items: int, q_off, q_len, k_off,
                           k_len, lq, lk, group):
        """``cross_block`` of every sequence at once: item i attends from its rows of ``x`` to its rows of ``ctxt``."""
        rows, D = x.shape
        xn, xnp = self.layernorm(x, blk.norm1, want_f32=True)
        _, cnp = self.layernorm(ctxt, blk.norm_context, want_f32=False)
        a = blk.cross_attn
        q, _ = self.linear(xnp, a.in_proj_weight, a.in_proj_bias, 0, D)
        kv, _ = self.linear(cnp, a.in_proj_weight, a.in_proj_bias, D, 3 * D)
        ctx = self.attention_varlen(q, kv[:, :D], kv[:, D:], H, D // H, step, items, q_off, q_len, k_off, k_len, lq, lk,
                                    group, rows, D, zero=lq[0] != lq[1])
        y, _ = self.linear(ctx, a.out_proj.weight, a.out_proj.bias, resid=xn)
        self.mlp_tail(y, blk, out=x)


# One forward is ~180 kernel launches (coarse tracker) whose device time is a few milliseconds at most: issued one by one
# from Python the host is the bottleneck, so the launch sequence of a (shape, precision) is captured once into a CUDA
# graph and replayed (workspaces live in the graph's private pool).  False = eager launches (A/B timing, debugging).
USE_CUDA_GRAPH = True
_MAX_GRAPHS = 4


class _Captured:
    """``counts`` given: the ragged forward, captured for the capacity of ``x`` (B, N_cap, T, Din); the track counts (and
    ``frames``, the frame counts) are read from device buffers, so one graph serves every set of counts up to N_cap
    (and T)."""

    def __init__(self, m, x: torch.Tensor, np_: int, counts: torch.Tensor = None, frames: torch.Tensor = None):
        self.x = torch.empty_like(x)
        self.x.copy_(x)
        self.counts = None if counts is None else counts.clone()
        self.frames = None if frames is None else frames.clone()
        run = (lambda: forward_eager(m, self.x, np_)) if counts is None else (
            lambda: forward_ragged_eager(m, self.x, np_, self.counts, self.frames))
        side = torch.cuda.Stream(device=x.device)
        side.wait_stream(torch.cuda.current_stream(x.device))
        with torch.cuda.stream(side):                      # warm-up: weight planes, kernel attributes, allocator
            run()
        torch.cuda.current_stream(x.device).wait_stream(side)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.out = run()

    def __call__(self, x: torch.Tensor, counts: torch.Tensor = None, frames: torch.Tensor = None) -> torch.Tensor:
        if counts is None:
            self.x.copy_(x, non_blocking=True)
        else:
            n = x.shape[1]
            self.x[:, :n].copy_(x, non_blocking=True)
            self.x[:, n:].zero_()
            self.counts.copy_(counts, non_blocking=True)
            if frames is not None:
                self.frames.copy_(frames, non_blocking=True)
        self.graph.replay()
        if counts is None:
            return self.out.clone()
        return self.out[:, :x.shape[1]].clone()


def _weights_tag(m) -> tuple:
    ps = list(m.parameters())
    return (ps[0].data_ptr(), sum(p._version for p in ps))


def forward(m, x: torch.Tensor, np_: int) -> torch.Tensor:
    """``EfficientUpdateFormer.forward`` (blocks.py:298-348) for tokens ``x`` (B, N, T, input_dim) float32 on CUDA."""
    if not USE_CUDA_GRAPH or torch.cuda.is_current_stream_capturing():
        return forward_eager(m, x, np_)
    if not hasattr(m, "_tc_graphs"):
        m._tc_graphs = {}
    key = (tuple(x.shape), np_, str(x.device), _weights_tag(m))
    g = m._tc_graphs.get(key)
    if g is None:
        while len(m._tc_graphs) >= _MAX_GRAPHS:
            m._tc_graphs.pop(next(iter(m._tc_graphs)))
        with torch.cuda.device(x.device):
            g = m._tc_graphs[key] = _Captured(m, x.contiguous(), np_)
        m._tc_captures = getattr(m, "_tc_captures", 0) + 1
    return g(x)


# Track capacity of a ragged graph: N_max rounded up to this, so that a dataset's changing counts reuse a few graphs.
RAGGED_TRACK_QUANTUM = 64


def ragged_supported(m) -> bool:
    """The varlen space attention serves problems with more than 32 queries or keys: true for >= 33 virtual tracks."""
    return not m.add_space_attn or m.num_virtual_tracks > 32


def forward_ragged(m, x: torch.Tensor, np_: int, counts: torch.Tensor, frames: torch.Tensor = None) -> torch.Tensor:
    """``EfficientUpdateFormer.forward`` of B sequences at once: tokens ``x`` (B, N_max, T, input_dim), ``counts`` (B,)
    int32 on the device (1 <= counts[b] <= N_max).  Sequence b's rows n < counts[b] get what the forward of that
    sequence alone gives; its rows n >= counts[b] are zeros.  ``frames`` (B,) int32 on the device (1 <= frames[b] <= T),
    or None: sequence b has frames[b] frames, and its rows of frames t >= frames[b] are zeros too.  ``counts=None`` with
    ``frames``: every sequence has N_max tracks (no track padding is added)."""
    B, N, T, Din = x.shape
    if counts is None:
        counts = torch.full((B,), N, dtype=torch.int32, device=x.device)
        ncap = N
    else:
        ncap = (N + RAGGED_TRACK_QUANTUM - 1) // RAGGED_TRACK_QUANTUM * RAGGED_TRACK_QUANTUM
    if not USE_CUDA_GRAPH or torch.cuda.is_current_stream_capturing():
        xp = x.new_zeros((B, ncap, T, Din))
        xp[:, :N] = x
        return forward_ragged_eager(m, xp, np_, counts, frames)[:, :N]
    if not hasattr(m, "_tc_graphs"):
        m._tc_graphs = {}
    key = ("ragged", B, ncap, T, Din, np_, str(x.device), _weights_tag(m)) + (() if frames is None else ("frames",))
    g = m._tc_graphs.get(key)
    if g is None:
        while len(m._tc_graphs) >= _MAX_GRAPHS:
            m._tc_graphs.pop(next(iter(m._tc_graphs)))
        xp = x.new_zeros((B, ncap, T, Din))
        xp[:, :N] = x
        with torch.cuda.device(x.device):
            g = m._tc_graphs[key] = _Captured(m, xp, np_, counts, frames)
        m._tc_captures = getattr(m, "_tc_captures", 0) + 1
    return g(x, counts, frames)


class _RaggedLayout:
    """Device index arrays of the space attention over B sequences: item i = (sequence b, frame t) = b * T + t.  Point
    rows are (b, n, t) -> (b * N_cap + n) * T + t, virtual rows (b, v, t) -> (b * V + v) * T + t of their own block.

    ``space_group``: the problem count that picks each space item's kernel family, the frame count of the single call.

    With ``frames`` (frame counts), the space items of frames t >= frames[b] have length 0 and choose their family for
    frames[b] problems, and the time attention is varlen too: item k = track k of the (points, then virtual tracks) row
    order, rows k * T + t for t < frames of its sequence; its kernel family is chosen for the problem count
    counts[b] + V of the single-sequence call."""

    def __init__(self, counts: torch.Tensor, B: int, ncap: int, V: int, T: int, frames: torch.Tensor = None):
        dev = counts.device
        b = torch.arange(B, device=dev, dtype=torch.int32).repeat_interleave(T)
        t = torch.arange(T, device=dev, dtype=torch.int32).repeat(B)
        self.items, self.V, self.ncap = B * T, V, ncap
        self.pts_off = (b * (ncap * T) + t).contiguous()
        self.vir_off = (b * (V * T) + t).contiguous()
        self.pts_len = counts.to(torch.int32).repeat_interleave(T).contiguous()
        self.vir_len = torch.full((B * T,), V, dtype=torch.int32, device=dev)
        self.vir_lq = (V, V)
        self.pts_lq = (1, ncap)
        self.space_group = T
        if frames is not None:
            live = (t < frames.to(torch.int32).repeat_interleave(T)).to(torch.int32)
            self.pts_len = (self.pts_len * live).contiguous()
            self.vir_len = (self.vir_len * live).contiguous()
            self.vir_lq = (0, V)
            self.pts_lq = (0, ncap)
            self.space_group = (frames.to(torch.int32).repeat_interleave(T).contiguous(), 1, T)
            seq = torch.cat([torch.arange(B, device=dev, dtype=torch.int32).repeat_interleave(ncap),
                             torch.arange(B, device=dev, dtype=torch.int32).repeat_interleave(V)])
            self.tracks = B * (ncap + V)
            self.trk_off = (torch.arange(self.tracks, device=dev, dtype=torch.int32) * T).contiguous()
            self.trk_len = frames.to(torch.int32)[seq].contiguous()
            self.trk_group = (counts.to(torch.int32)[seq] + V).contiguous()
            self.trk_grange = (1 + V, ncap + V)


def forward_ragged_eager(m, x: torch.Tensor, np_: int, counts: torch.Tensor, frames: torch.Tensor = None) -> torch.Tensor:
    """Ragged forward for x (B, N_cap, T, input_dim).  Tokens are laid out as all sequences' point rows followed by all
    sequences' virtual rows, so every LayerNorm and GEMM of a block is one launch over all sequences and the space
    attention is one varlen launch per kernel family.  Padded point rows are never keys or queries of the space
    attention; they only pass through row-wise work (and the time attention, per track) and stay finite."""
    B, Nc, T, Din = x.shape
    D, H, V = m.hidden_size, m.num_heads, (m.num_virtual_tracks if m.add_space_attn else 0)
    if not hasattr(m, "_tc_weights"):
        m._tc_weights = _Weights()
    with torch.cuda.device(x.device):
        run = _Run(m._tc_weights, np_, x.device)
        x = x.contiguous()
        P = B * Nc * T
        xp = run.split(x.view(P, Din))
        skip, _ = run.linear(xp, m.input_transform.weight, m.input_transform.bias)          # (B*Nc*T, D)
        flat = torch.empty((P + B * V * T, D), dtype=torch.float32, device=x.device)
        flat[:P] = skip
        pts, vir = flat[:P], flat[P:]
        if V:
            vir.view(B, V, T, D)[:] = m.virual_tracks                                        # (1, V, 1, D) broadcast
        lay = _RaggedLayout(counts, B, Nc, V, T, frames) if V or frames is not None else None
        every = len(m.time_blocks) // len(m.space_virtual_blocks) if V else 0
        j = 0
        for i, tb in enumerate(m.time_blocks):
            if frames is None:
                run.self_block(flat, tb, B * (Nc + V), T, T, 1, H)                           # time attention per track
            else:
                run.self_block_varlen(flat, tb, H, 1, lay.tracks, lay.trk_off, lay.trk_len, (1, T),
                                      (lay.trk_group, *lay.trk_grange))
            if V and i % every == 0:
                run.cross_block_varlen(vir, pts, m.space_virtual2point_blocks[j], H, T, lay.items, lay.vir_off, lay.vir_len,
                                       lay.pts_off, lay.pts_len, lay.vir_lq, lay.pts_lq, lay.space_group)
                run.self_block_varlen(vir, m.space_virtual_blocks[j], H, T, lay.items, lay.vir_off, lay.vir_len, lay.vir_lq,
                                      lay.space_group)
                run.cross_block_varlen(pts, vir, m.space_point2virtual_blocks[j], H, T, lay.items, lay.pts_off, lay.pts_len,
                                       lay.vir_off, lay.vir_len, lay.pts_lq, lay.vir_lq, lay.space_group)
                j += 1
        sp = run.new_planes(P, D)
        _lib.check(lib.comet_add_planes_f32(pts.data_ptr(), skip.data_ptr(), sp.data_ptr(), sp.stride(0), np_, P * D,
                                            run.stream))
        out, _ = run.linear(sp, m.flow_head.weight, m.flow_head.bias)
        out = out.view(B, Nc, T, -1)
        real = torch.arange(Nc, device=x.device)[None, :] < counts[:, None]
        if frames is None:
            return out.masked_fill_(~real[:, :, None, None], 0.0)
        live = torch.arange(T, device=x.device)[None, :] < frames[:, None]                    # (B, T)
        return out.masked_fill_(~(real[:, :, None] & live[:, None, :])[..., None], 0.0)


def forward_eager(m, x: torch.Tensor, np_: int) -> torch.Tensor:
    B, N, T, Din = x.shape
    D, H, V = m.hidden_size, m.num_heads, (m.num_virtual_tracks if m.add_space_attn else 0)
    if not hasattr(m, "_tc_weights"):
        m._tc_weights = _Weights()
    with torch.cuda.device(x.device):
        run = _Run(m._tc_weights, np_, x.device)
        x = x.contiguous()
        xp = run.split(x.view(B * N * T, Din))
        skip, _ = run.linear(xp, m.input_transform.weight, m.input_transform.bias)          # (B*N*T, D)
        if V:
            tok = torch.empty((B, N + V, T, D), dtype=torch.float32, device=x.device)
            tok[:, :N] = skip.view(B, N, T, D)
            tok[:, N:] = m.virual_tracks                                                     # (1, V, 1, D) broadcast over B, T
        else:
            tok = skip.clone().view(B, N, T, D)
        flat = tok.view(B * (N + V) * T, D)
        every = len(m.time_blocks) // len(m.space_virtual_blocks) if V else 0
        j = 0
        for i, tb in enumerate(m.time_blocks):
            run.self_block(flat, tb, B * (N + V), T, T, 1, H)                                # time attention per track
            if V and i % every == 0:
                for b in range(B):
                    pts = tok[b, :N].view(N * T, D)
                    vir = tok[b, N:].view(V * T, D)
                    run.cross_block(vir, pts, m.space_virtual2point_blocks[j], T, H)
                    run.self_block(vir, m.space_virtual_blocks[j], T, V, 1, T, H)            # over the virtual tracks, per frame
                    run.cross_block(pts, vir, m.space_point2virtual_blocks[j], T, H)
                j += 1
        pts_all = tok[:, :N].reshape(B * N * T, D)          # a view unless B > 1 with virtual tracks in between
        sp = run.new_planes(B * N * T, D)
        _lib.check(lib.comet_add_planes_f32(pts_all.data_ptr(), skip.data_ptr(), sp.data_ptr(), sp.stride(0), np_, B * N * T * D,
                                            run.stream))
        out, _ = run.linear(sp, m.flow_head.weight, m.flow_head.bias)
        return out.view(B, N, T, -1)
