"""Sequences of different image sizes in one ``track_batch`` call (``image_sizes=`` / a list of clips of different sizes,
size groups, the packed frame buffer and the packed patch encoder).  Contract: sequence b gets what ``track`` returns
for it alone on its own clip, in its own pixel coordinates; ``num_tracks``, ``num_frames`` and ``query_frames`` compose
with it; equal sizes run the one-size path unchanged.

Kernel-level results are held bitwise to the same kernels on each sequence's own contiguous frames; loop-level results
to the float64 reference with the bars of test_full_size.py, and to per-sequence ``track`` calls at iteration 0."""
import contextlib
from types import SimpleNamespace as NS

import pytest
import torch
import torch.nn as nn

import cases
from conftest import rel_to_max

SPEC = 1e-4


def cfg():
    return NS(track_conf=False, MODEL=NS(TRACK=NS(efficient_corr=False)))


def load_seeded(module, seed):
    sd = cases.seeded_state_dict({k: tuple(v.shape) for k, v in module.state_dict().items()}, seed)
    module.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()}, strict=True)
    return module


def bar(ref32, ref64):
    return max(SPEC, 3.0 * rel_to_max(ref32, ref64))


def swap(x, q, dim=1):
    order = list(range(x.shape[dim]))
    order[0], order[q] = q, 0
    return x.index_select(dim, torch.tensor(order, device=x.device))


def padded(clips, fill=float("nan")):
    """A (B, S_max, 3, H_max, W_max) tensor holding the clips, ``fill`` everywhere else."""
    S = max(c.shape[0] for c in clips)
    H = max(c.shape[2] for c in clips)
    W = max(c.shape[3] for c in clips)
    out = clips[0].new_full((len(clips), S, 3, H, W), fill)
    for b, c in enumerate(clips):
        out[b, :c.shape[0], :, :c.shape[2], :c.shape[3]] = c
    return out


def sizes_of(clips):
    return torch.tensor([[c.shape[2], c.shape[3]] for c in clips])


# ------------------------------------------------------------------------------------------------ CPU
def _stub_tracker():
    """A TrackerPredictor whose coarse predictor is the real ``BaseTrackerPredictor.forward`` for the size-group and
    frame-table handling (on the CPU it runs each group alone and gathers the maps) around a cheap computation that
    depends on the maps' size, values and frame order."""
    import comet_pose_estimation_b200 as cb

    class Stub(cb.BaseTrackerPredictor):
        def forward(self, query_points, fmaps=None, iters=4, return_feat=False, down_ratio=1, is_train=False,
                    track_feats=None, TRACKorPOSE=True, ind=0, num_tracks=None, num_frames=None, frame_index=None,
                    group_items=None):
            if frame_index is not None or isinstance(fmaps, list):
                return super().forward(query_points, fmaps, iters, return_feat, down_ratio, is_train, track_feats,
                                       TRACKorPOSE, ind, num_tracks, num_frames, frame_index, group_items)
            B, S = fmaps.shape[:2]
            N = query_points.shape[1]
            m = fmaps.mean(dim=(2, 3, 4)) + fmaps.shape[-1] * 1e-3                # (B, S), size-dependent
            live = torch.ones(B, S, N, dtype=torch.bool)
            if num_frames is not None:
                live &= (torch.arange(S)[None, :] < torch.tensor(list(num_frames))[:, None])[..., None]
            if num_tracks is not None:
                live &= (torch.arange(N)[None, :] < torch.tensor(list(num_tracks))[:, None])[:, None, :]
            c = query_points[:, None] * (1.0 + m[..., None, None]) + m[:, :1, None, None] * torch.arange(S)[None, :, None, None]
            c = c * live[..., None]
            vis = torch.sigmoid(c.sum(-1)) * live
            return [c * 0.5, c], vis, None, None, None

    torch.manual_seed(0)
    return cb.TrackerPredictor(coarse_fnet=nn.Conv2d(3, 4, 1), coarse_predictor=Stub(cfg=cfg()),
                               coarse_down_ratio=1).eval()


def test_min_image_size():
    """The floor follows from the pyramid and the patch: 5 levels of stride-4 maps of a half-size image need 16x16 maps,
    so 128 pixels; the stub (no down-sampling) needs 64."""
    import comet_pose_estimation_b200 as cb

    assert cb.TrackerPredictor().min_image_size() == 128
    assert cb.TrackerPredictor(coarse_down_ratio=1).min_image_size() == 64
    assert cb.TrackerPredictor(coarse_down_ratio=1).min_image_size(fine_tracking=True) == 64
    tp = cb.TrackerPredictor(coarse_down_ratio=1, coarse_predictor=cb.BaseTrackerPredictor(corr_levels=2, cfg=cfg()))
    assert tp.min_image_size(fine_tracking=False) == 8 and tp.min_image_size() == 31


def _bad_calls():
    g = torch.Generator().manual_seed(0)
    clips = [torch.rand(3, 3, 64, 80, generator=g), torch.rand(2, 3, 72, 64, generator=g)]
    pad = padded(clips, 0.0)
    ok = sizes_of(clips)
    return [(pad, dict(image_sizes=ok[:1])),                                  # (1, 2) for two sequences
            (pad, dict(image_sizes=torch.tensor([[64, 80, 1], [72, 64, 1]]))),  # (B, 3)
            (pad, dict(image_sizes=ok.float())),                              # not integers
            (pad, dict(image_sizes=[[64.0, 80.5], [72, 64]])),                # not integers (nested lists)
            (pad, dict(image_sizes=torch.tensor([[64, 81], [72, 64]]))),      # wider than the padded tensor
            (pad, dict(image_sizes=torch.tensor([[64, 80], [73, 64]]))),      # taller than the padded tensor
            (clips, dict(image_sizes=torch.tensor([[64, 80], [64, 72]]))),    # list and sizes disagree
            (pad, dict(image_sizes=torch.tensor([[64, 80], [72, 63]]))),      # below the floor (64 for the stub)
            ([clips[0], torch.rand(2, 3, 63, 64, generator=g)], {}),          # a list below the floor
            (pad, dict(image_sizes=torch.tensor([[0, 80], [72, 64]])))]       # not positive


@pytest.mark.parametrize("k", range(10))
def test_invalid_image_sizes_are_refused(k):
    tp = _stub_tracker()
    images, kw = _bad_calls()[k]
    qs = [torch.zeros(3, 2), torch.zeros(4, 2)]
    with pytest.raises(AssertionError):
        tp.track_batch(images, qs, fine_tracking=False, **kw)


def _mixed_clips(g, frames=(4, 3, 4, 2), sizes=((64, 96), (80, 64), (64, 96), (64, 64))):
    return [torch.rand(s, 3, h, w, generator=g) for s, (h, w) in zip(frames, sizes)]


@pytest.mark.parametrize("mode", ["plain", "num_frames", "query_frames"])
def test_cpu_mixed_sizes_equal_per_sequence_calls(mode):
    """The CPU definition: a mixed batch equals per-sequence calls on each sequence's own clip, padded back."""
    import comet_pose_estimation_b200 as cb

    tp = _stub_tracker()
    g = torch.Generator().manual_seed(1)
    clips = _mixed_clips(g, frames=(4, 4, 4, 4) if mode == "plain" else (4, 3, 4, 2))
    qs = [torch.rand(n, 2, generator=g) * 60 for n in (5, 2, 4, 3)]
    kw = {}
    if mode == "query_frames":
        kw["query_frames"] = [torch.tensor([0, 3, 3, 1, 0]), torch.tensor([2, 1]), torch.tensor([0, 0, 0, 0]),
                              torch.tensor([1, 0, 1])]
    with torch.no_grad():
        if mode == "plain":
            out = tp.track_batch(padded(clips), qs, fine_tracking=False, image_sizes=sizes_of(clips))
        else:
            out = tp.track_batch(padded(clips), qs, fine_tracking=False, image_sizes=sizes_of(clips),
                                 num_frames=[c.shape[0] for c in clips], **kw)
        assert out["image_sizes"].tolist() == sizes_of(clips).tolist() and out["image_sizes"].dtype == torch.int64
        S = max(c.shape[0] for c in clips)
        parts = cb.split_batch(out)
        for b, (c, q) in enumerate(zip(clips, qs)):
            n, s = q.shape[0], c.shape[0]
            qf = kw.get("query_frames", [None] * 4)[b]
            one = tp.track(c[None], q[None], fine_tracking=False, query_frames=qf)
            assert set(parts[b]) == set(one)
            for k in ("coarse_pred_track", "vis", "pred_score", "refine_pred_track"):
                assert parts[b][k].shape == one[k].shape, k
                assert torch.allclose(parts[b][k], one[k], rtol=1e-6, atol=1e-6), (k, b)
                assert torch.count_nonzero(out[k][b, s:]) == 0 and torch.count_nonzero(out[k][b, :, n:]) == 0
            for i, lvl in enumerate(out["coarse_pred_track_list"]):
                assert torch.allclose(lvl[b:b + 1, :s, :n], one["coarse_pred_track_list"][i], rtol=1e-6, atol=1e-6)
            assert out["coarse_pred_track"].shape[1] == S


def test_cpu_list_equals_padded_with_nan():
    tp = _stub_tracker()
    g = torch.Generator().manual_seed(2)
    clips = _mixed_clips(g)
    qs = [torch.rand(n, 2, generator=g) * 60 for n in (5, 2, 4, 3)]
    with torch.no_grad():
        a = tp.track_batch(clips, qs, fine_tracking=False)
        b = tp.track_batch(padded(clips), qs, fine_tracking=False, image_sizes=sizes_of(clips),
                           num_frames=[c.shape[0] for c in clips])
    assert set(a) == set(b)
    for k, v in a.items():
        if isinstance(v, torch.Tensor):
            assert torch.equal(v, b[k]), k
            assert not v.is_floating_point() or torch.isfinite(v).all(), k


def test_cpu_equal_sizes_run_the_one_size_path():
    tp = _stub_tracker()
    g = torch.Generator().manual_seed(3)
    images = torch.rand(3, 4, 3, 64, 80, generator=g)
    qs = [torch.rand(n, 2, generator=g) * 60 for n in (5, 2, 4)]
    with torch.no_grad():
        want = tp.track_batch(images, qs, fine_tracking=False)
        via_sizes = tp.track_batch(images, qs, fine_tracking=False, image_sizes=[[64, 80]] * 3)
        via_list = tp.track_batch(list(images), qs, fine_tracking=False, image_sizes=[[64, 80]] * 3)
        big = torch.full((3, 4, 3, 70, 90), float("nan"))
        big[..., :64, :80] = images
        cropped = tp.track_batch(big, qs, fine_tracking=False, image_sizes=[[64, 80]] * 3)
    for got in (via_sizes, via_list, cropped):
        assert got["image_sizes"].tolist() == [[64, 80]] * 3
        for k, v in want.items():
            if isinstance(v, torch.Tensor) and k != "num_frames":
                assert torch.equal(v, got[k]), k


def _input_forms():
    """(images, keywords, extra keys, frame axis) of every input form of ``track_batch``: a one-size tensor keeps its
    S_max whatever ``num_frames`` says; lists, mixed sizes and ``clip_frames`` give max(S_b)."""
    g = torch.Generator().manual_seed(5)
    c = lambda s, h=64, w=80: torch.rand(s, 3, h, w, generator=g)  # noqa: E731
    T = torch.rand(3, 8, 3, 64, 80, generator=g)
    zero = [torch.zeros(n, dtype=torch.int64) for n in (5, 2, 4)]
    qf = [torch.tensor([0, 1, 1, 0, 2]), torch.tensor([0, 0]), torch.tensor([3, 0, 0, 0])]
    equal, cropped, mixed = [[64, 80]] * 3, [[64, 72]] * 3, [[64, 80], [64, 72], [64, 80]]
    nt, nf, nfq, ns = {"num_tracks"}, {"num_frames", "num_tracks"}, {"num_tracks", "query_frames"}, {"image_sizes", "num_tracks"}
    nsf = ns | {"num_frames"}
    return {"tensor": (T, {}, nt, 8),
            "tensor_full_frames": (T, dict(num_frames=[8, 8, 8]), nf, 8),
            "tensor_ragged_frames": (T, dict(num_frames=[6, 3, 5]), nf, 8),
            "tensor_zero_query_frames": (T, dict(query_frames=zero), nfq, 8),
            "tensor_query_frames": (T, dict(query_frames=qf), nfq, 8),
            "tensor_query_frames_ragged_frames": (T, dict(query_frames=qf, num_frames=[6, 3, 5]), nfq | nf, 8),
            "tensor_equal_sizes": (T, dict(image_sizes=equal), ns, 8),
            "tensor_equal_sizes_cropped": (T, dict(image_sizes=cropped), ns, 8),
            "tensor_mixed_sizes": (T, dict(image_sizes=mixed), nsf, 8),
            "tensor_mixed_sizes_ragged_frames": (T, dict(image_sizes=mixed, num_frames=[6, 3, 5]), nsf, 6),
            "list_equal": ([c(4), c(4), c(4)], {}, nf, 4),
            "list_equal_sizes": ([c(4), c(4), c(4)], dict(image_sizes=equal), nsf, 4),
            "list_ragged_frames": ([c(6), c(3), c(5)], {}, nf, 6),
            "list_mixed_sizes": ([c(4), c(3, 72, 64), c(4)], {}, nsf, 4),
            "clip_frames_one_size": (c(10), dict(clip_frames=[[0, 1, 2], [2, 3], [5, 5, 1, 0]]), nf, 4),
            "clip_frames_two_sizes": ([c(5), c(4, 72, 64)], dict(clip_frames=[[0, 1, 2], [5, 6], [8, 7, 6, 5]]), nsf, 4)}


@pytest.mark.parametrize("form", list(_input_forms()))
def test_cpu_keys_and_frame_axis_of_every_input_form(form):
    tp = _stub_tracker()
    images, kw, extra, S = _input_forms()[form]
    qs = [torch.rand(n, 2, generator=torch.Generator().manual_seed(n)) * 60 for n in (5, 2, 4)]
    with torch.no_grad():
        out = tp.track_batch(images, qs, fine_tracking=False, **kw)
    assert set(out) == {"coarse_pred_track_list", "coarse_pred_track", "vis", "conf", "refine_pred_track",
                        "pred_score"} | extra
    assert out["coarse_pred_track"].shape == (3, S, 5, 2)


def test_packed_frames_builder():
    import comet_pose_estimation_b200 as cb

    g = torch.Generator().manual_seed(4)
    clips = [torch.rand(s, 3, h, w, generator=g) for s, (h, w) in zip((3, 2, 4, 1), ((48, 64), (40, 40), (48, 64), (40, 56)))]
    big = padded(clips)                                                    # NaN outside every clip
    views = [big[b, :c.shape[0], :, :c.shape[2], :c.shape[3]] for b, c in enumerate(clips)]
    pk = cb.PackedFrames(views)
    # groups by increasing (H, W), sequences of a group in batch order
    assert pk.groups == [((40, 40), [1]), ((40, 56), [3]), ((48, 64), [0, 2])]
    assert pk.seq_first == [3, 0, 6, 2] and pk.seq_frames == [3, 2, 4, 1]
    assert pk.group_first == [0, 2, 3] and pk.group_frames == [2, 1, 7]
    hw = [(40, 40)] * 2 + [(40, 56)] + [(48, 64)] * 7
    assert pk.frame_hw.tolist() == [list(x) for x in hw] and pk.frame_hw.dtype == torch.int32
    off = [0]
    for h, w in hw[:-1]:
        off.append(off[-1] + 3 * h * w)
    assert pk.frame_offset.tolist() == off and pk.frame_offset.dtype == torch.int64
    assert pk.data.numel() == sum(c.numel() for c in clips) and pk.num_frames == 10
    assert torch.isfinite(pk.data).all()                                   # nothing outside [:S_b, :, :H_b, :W_b] read
    for b, c in enumerate(clips):
        assert torch.equal(pk.clip(b), c)
        assert pk.clip(b).data_ptr() == pk.data.data_ptr() + 4 * off[pk.seq_first[b]]   # a view, no copy
    assert torch.equal(pk.group(2), torch.cat([clips[0], clips[2]]))
    assert pk.group(2).data_ptr() == pk.data.data_ptr() + 4 * off[3]


def test_split_batch_drops_image_sizes():
    import comet_pose_estimation_b200 as cb

    B, S, N = 3, 5, 7
    counts, frames = [7, 1, 4], [5, 2, 1]
    t = lambda *s: torch.randn(*s)  # noqa: E731
    out = {"coarse_pred_track_list": [t(B, S, N, 2) for _ in range(4)], "coarse_pred_track": t(B, S, N, 2),
           "vis": t(B, S, N), "conf": None, "refine_pred_track": t(B, S, N, 2), "track_score": t(B, S, N),
           "pred_score": t(B, S, N), "num_tracks": torch.tensor(counts), "num_frames": torch.tensor(frames),
           "image_sizes": torch.tensor([[128, 128], [384, 512], [256, 128]])}
    for p, n, s in zip(cb.split_batch(out), counts, frames):
        assert set(p) == set(out) - {"num_tracks", "num_frames", "image_sizes"}
        assert p["coarse_pred_track"].shape == (1, s, n, 2) and p["vis"].shape == (1, s, n)


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture
def no_tf32():
    a, b = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = a, b


def _guarded(clips, gap=4099):
    """A packed buffer of the clips' frames with NaN guard bands of ``gap`` elements before, between and after the
    frames (the offset table allows gaps): a read outside a frame turns its map to NaN."""
    offs, hws, parts, at = [], [], [], gap
    nan = lambda n: torch.full((n,), float("nan"), device="cuda")  # noqa: E731
    parts.append(nan(gap))
    for c in clips:
        for f in c:
            offs.append(at)
            hws.append(tuple(f.shape[1:]))
            parts.append(f.reshape(-1))
            parts.append(nan(gap))
            at += f.numel() + gap
    off = torch.tensor(offs, dtype=torch.int64, device="cuda")
    hw = torch.tensor(hws, dtype=torch.int32, device="cuda")
    return NS(data=torch.cat(parts), device=torch.device("cuda"), num_frames=len(offs), device_tables=lambda: (off, hw))


@pytest.mark.gpu
def test_packed_encoder_matches_indexed_encoder_per_clip(no_tf32):
    """The packed patch encoder == ``comet_shallow_encoder_from_images_indexed_f32`` on each sequence's own contiguous
    clip, bit for bit, for patches clamped at all four borders of small and non-square frames, with frame counts and
    swapped frame tables; padded frames are zeros and nothing outside a frame is read."""
    import comet_pose_estimation_b200 as cb
    from comet_pose_estimation_b200.utils import query_frame_items

    fnet = load_seeded(cb.ShallowEncoder(input_dim=3).eval(), 3).cuda()
    g = torch.Generator(device="cuda").manual_seed(2)
    S = 5
    frames, sizes = [5, 3, 4, 5], [(31, 31), (40, 33), (64, 48), (96, 128)]
    clips = [torch.randn(s, 3, h, w, device="cuda", generator=g) for s, (h, w) in zip(frames, sizes)]
    firsts = [sum(frames[:b]) for b in range(len(frames))]
    items, fi = query_frame_items([[0, 3, 3], [1, 0], [0], [4, 2, 0]], frames, S)
    src = fi - torch.tensor([b * S for b, _, _ in items])[:, None]
    table = torch.stack([firsts[b] + src[i].clamp(max=frames[b] - 1) for i, (b, _, _) in enumerate(items)]).cuda()
    counts = [3, 2, 4, 1, 2, 1, 3, 2]
    assert len(counts) == len(items)
    nf = torch.tensor([frames[b] for b, _, _ in items], dtype=torch.int32, device="cuda")
    seq = torch.tensor([i for i, n in enumerate(counts) for _ in range(n)], device="cuda")
    P = len(seq)
    # corners from 40 pixels before to 40 past every border of the track's own frame
    hw = torch.tensor([sizes[items[i][0]] for i in seq.tolist()], device="cuda")
    u = torch.rand(P, S, 2, device="cuda", generator=g)
    tl = (u * (hw.flip(-1)[:, None, :] + 80) - 40).floor().int()
    tl[0, :, 0], tl[1, :, 1] = -40, 10_000                                   # every border reached
    pk = _guarded(clips)
    with torch.no_grad():
        got, _ = fnet.encode_packed_frames_patches_of(pk, tl, seq, num_frames=nf, frame_index=table)
    got = got.permute(0, 2, 3, 1).reshape(P, S, 16, 16, 32)
    live = torch.arange(S, device="cuda")[None, :] < nf[seq][:, None]
    assert torch.isfinite(got).all() and torch.count_nonzero(got[~live]) == 0
    for i, (b, _, _) in enumerate(items):
        mine = (seq == i).nonzero()[:, 0]
        images = torch.full((1, S, 3) + sizes[b], float("nan"), device="cuda")
        images[0, :frames[b]] = clips[b]
        local = (table[i:i + 1] - firsts[b]).clamp(min=0)
        with torch.no_grad():
            want, _ = fnet.encode_packed_patches_of(images, tl[mine], torch.zeros_like(mine), num_frames=nf[i:i + 1],
                                                    frame_index=local)
        assert torch.equal(got[mine], want.permute(0, 2, 3, 1).reshape(len(mine), S, 16, 16, 32)), i


def _coarse_model():
    import comet_pose_estimation_b200 as cb

    return load_seeded(cb.BaseTrackerPredictor(cfg=cfg(), **cases.FULL_COARSE_CTOR).eval(), cases.FULL_SEEDS["coarse"]).cuda()


def _fine_models():
    import comet_pose_estimation_b200 as cb

    fnet = load_seeded(cb.ShallowEncoder(input_dim=3).eval(), cases.FULL_SEEDS["fnet"]).cuda()
    ftr = load_seeded(cb.BaseTrackerPredictor(cfg=cfg(), **cases.FULL_FINE_CTOR).eval(), cases.FULL_SEEDS["fine"]).cuda()
    return fnet.to(memory_format=torch.channels_last), ftr


def _group_case(g, ragged, S=8):
    """Three size groups (maps 48x48, 64x64 -- the tensor path -- and 60x80): per-group maps, items, counts, frame
    counts and (``ragged``) a swapped frame table per group."""
    from comet_pose_estimation_b200.utils import query_frame_items

    shapes = [(2, 48, 48), (2, 64, 64), (1, 60, 80)]
    fmaps = [torch.randn(n, S, 128, h, w, device="cuda", generator=g) for n, h, w in shapes]
    if not ragged:
        return fmaps, [n for n, _, _ in shapes], None, None, [[300, 37], [512, 64], [100]]
    frames = [[8, 5], [8, 6], [7]]
    qf = [[[0, 3], [1, 1]], [[0, 7], [5]], [[2, 0]]]
    for f, fr in zip(fmaps, frames):
        for j, s in enumerate(fr):
            f[j, s:] = 0.0
    tables, items_per_group, item_frames = [], [], []
    for fr, q in zip(frames, qf):
        items, fi = query_frame_items(q, fr, S)
        tables.append(fi)
        items_per_group.append(len(items))
        item_frames += [fr[b] for b, _, _ in items]
    counts = [[300, 37, 5], [512, 64, 200], [100, 1]]
    return fmaps, items_per_group, torch.cat(tables), item_frames, counts


@pytest.mark.gpu
@pytest.mark.parametrize("ragged", [False, True])
@pytest.mark.parametrize("autocast", [False, True])
def test_coarse_forward_with_size_groups_equals_per_group_calls(no_tf32, ragged, autocast):
    """Tokens bitwise equal to the per-group tokenizer, the first transformer pass (iteration 0) bitwise equal to the
    per-group forward, the whole loop within 1e-5."""
    import comet_pose_estimation_b200 as cb

    m = _coarse_model()
    g = torch.Generator(device="cuda").manual_seed(3)
    fmaps, group_items, fi, frames, counts = _group_case(g, ragged)
    counts = [n for c in counts for n in c]
    Bi, N, S = len(counts), max(counts), fmaps[0].shape[1]
    bounds = [sum(group_items[:k]) for k in range(len(group_items) + 1)]
    q = torch.rand(Bi, N, 2, device="cuda", generator=g)
    for k, f in enumerate(fmaps):
        q[bounds[k]:bounds[k + 1]] *= torch.tensor([f.shape[-1], f.shape[-2]], device="cuda") * 8.0
    tdim = m.transformer_dim
    coords = (q / 8.0)[:, None].repeat(1, S, 1, 1) + torch.randn(Bi, S, N, 2, device="cuda", generator=g)
    feats = torch.randn(Bi, S, N, 128, device="cuda", generator=g)
    kw = dict(num_tracks=counts, num_frames=frames)
    ctx = torch.autocast("cuda", dtype=torch.bfloat16) if autocast else contextlib.nullcontext()
    with ctx, torch.no_grad():
        blocks = [cb.CorrBlock(f, num_levels=5, radius=4) for f in fmaps]
        assert [b._pyr.split is not None for b in blocks] == [False, bool(cb._lib.lib.comet_has_tensor_path()), False]
        got = cb.TrackTokenizer(blocks, coords[:, 0], tdim, frame_index=fi, group_items=group_items, **kw).tokens(
            coords, feats).clone()
        for k, blk in enumerate(blocks):
            r0, r1 = bounds[k], bounds[k + 1]
            want = cb.TrackTokenizer(blk, coords[r0:r1, 0], tdim, num_tracks=counts[r0:r1],
                                     num_frames=None if frames is None else frames[r0:r1],
                                     frame_index=None if fi is None else fi[r0:r1]).tokens(coords[r0:r1], feats[r0:r1])
            assert torch.equal(got[r0:r1], want), k
        out = m(query_points=q, fmaps=fmaps, iters=3, return_feat=True, down_ratio=2, TRACKorPOSE=False, frame_index=fi,
                group_items=group_items, **kw)
        for k, f in enumerate(fmaps):
            r0, r1 = bounds[k], bounds[k + 1]
            one = m(query_points=q[r0:r1], fmaps=f, iters=3, return_feat=True, down_ratio=2, TRACKorPOSE=False,
                    num_tracks=counts[r0:r1], num_frames=None if frames is None else frames[r0:r1],
                    frame_index=None if fi is None else fi[r0:r1])
            assert torch.equal(out[0][0][r0:r1], one[0][0]), k
            for a, b in zip(out[0][1:], one[0][1:]):
                assert rel_to_max(a[r0:r1].cpu(), b.cpu()) <= 1e-5, k
            # vis is a bf16 output under autocast: a 1e-5 change of its float32 input can move it by one bf16 step
            vis_tol = 1e-5 if one[1].dtype == torch.float32 else 2.0 ** -8
            assert rel_to_max(out[1][r0:r1].float().cpu(), one[1].float().cpu()) <= vis_tol, k
    assert all(torch.isfinite(p).all() for p in out[0])


@pytest.mark.gpu
def test_golden_coarse_case_inside_size_groups(golden, no_tf32):
    g = golden("tracker_full")
    m = _coarse_model()
    fmaps, q = cases.tracker_case(**cases.FULL_COARSE_CASE)
    fmaps, q = torch.from_numpy(fmaps).cuda(), torch.from_numpy(q).cuda()
    S, N = fmaps.shape[1], q.shape[1]
    scale = cases.FULL_COARSE_CASE["down_ratio"] * 4
    gen = torch.Generator(device="cuda").manual_seed(9)
    small = torch.randn(1, S, 128, 48, 48, device="cuda", generator=gen)          # a 384x384 sequence
    wide = torch.randn(1, S, 128, 60, 80, device="cuda", generator=gen)           # a 480x640 sequence
    qp = torch.rand(3, N, 2, device="cuda", generator=gen) * scale * 0.9
    qp[0] *= 48
    qp[1] = q[0]
    qp[2] *= torch.tensor([80, 60], device="cuda")
    counts = [137, N, 300]
    with torch.no_grad():
        preds, vis, _, _, _ = m(query_points=qp, fmaps=[small, fmaps, wide], iters=cases.FULL_COARSE_ITERS,
                                return_feat=True, down_ratio=cases.FULL_COARSE_CASE["down_ratio"], TRACKorPOSE=False,
                                num_tracks=counts)
    for i in range(cases.FULL_COARSE_ITERS):
        assert rel_to_max(preds[i][1:2].cpu().numpy(), g[f"pred64_{i}"]) <= bar(g[f"pred32_{i}"], g[f"pred64_{i}"]), i
    assert rel_to_max(vis[1:2].cpu().numpy(), g["vis64"]) <= bar(g["vis32"], g["vis64"])
    assert all(torch.isfinite(p).all() for p in preds)


@pytest.mark.gpu
def test_golden_refine_case_inside_size_groups(golden, no_tf32):
    import comet_pose_estimation_b200 as cb

    r = golden("refine_full")
    fnet, ftr = _fine_models()
    images, _ = cases.refine_case(**cases.FULL_REFINE_CASE)
    images = torch.from_numpy(images).cuda()
    coarse = torch.from_numpy(r["coarse_pred"]).cuda()
    S, N = coarse.shape[1], coarse.shape[2]
    g = torch.Generator(device="cuda").manual_seed(4)
    clips = [torch.rand(S, 3, 384, 384, device="cuda", generator=g), images[0],
             torch.rand(S, 3, 480, 640, device="cuda", generator=g)]
    pk = cb.PackedFrames(clips)
    counts = [137, N, 300]
    batch_c = torch.zeros(3, S, N, 2, device="cuda")
    batch_c[1] = coarse[0]
    for i, (h, w) in ((0, (384, 384)), (2, (480, 640))):
        batch_c[i, :, :counts[i]] = torch.rand(S, counts[i], 2, device="cuda", generator=g) * torch.tensor(
            [w + 20.0, h + 20.0], device="cuda") - 10.0
    table = torch.stack([pk.seq_first[b] + torch.arange(S) for b in range(3)]).cuda()
    with torch.no_grad():
        refined, score = cb.refine_track(pk, fnet, ftr, batch_c, compute_score=True, num_tracks=counts, frame_index=table)
    inv = cb.inverted_score(score[1:2])
    for k, got in (("refined", refined[1:2]), ("score", score[1:2]), ("inverted", inv)):
        assert rel_to_max(got.cpu().numpy(), r[k + "64"]) <= bar(r[k + "32"], r[k + "64"]), k
    assert torch.isfinite(refined).all() and torch.isfinite(score).all()


def _tracker():
    import comet_pose_estimation_b200 as cb

    torch.manual_seed(0)
    return cb.TrackerPredictor().eval().cuda()


def _same(a, b, k):
    if isinstance(a, list):
        assert all(torch.equal(x, y) for x, y in zip(a, b)), k
    elif a is None:
        assert b is None, k
    else:
        assert torch.equal(a, b), k


@pytest.mark.gpu
def test_equal_sizes_are_bit_identical_to_no_sizes(no_tf32):
    tp = _tracker()
    g = torch.Generator(device="cuda").manual_seed(8)
    images = torch.randn(3, 6, 3, 256, 256, device="cuda", generator=g)
    qs = [torch.rand(n, 2, device="cuda", generator=g) * 240 for n in (90, 7, 200)]
    a = tp.track_batch(images, qs, coarse_iters=2)
    b = tp.track_batch(images, qs, coarse_iters=2, image_sizes=[[256, 256]] * 3)
    c = tp.track_batch(list(images), qs, coarse_iters=2, image_sizes=torch.tensor([[256, 256]] * 3))
    assert set(b) == set(a) | {"image_sizes"} and b["image_sizes"].tolist() == [[256, 256]] * 3
    for k in a:
        _same(a[k], b[k], k)
        if k != "num_frames":
            _same(a[k], c[k], k)


@pytest.mark.gpu
def test_padded_input_with_nan_equals_list_of_clips(no_tf32):
    tp = _tracker()
    g = torch.Generator(device="cuda").manual_seed(5)
    frames, sizes = [6, 4, 5], [(256, 256), (128, 192), (192, 160)]
    clips = [torch.randn(s, 3, h, w, device="cuda", generator=g) for s, (h, w) in zip(frames, sizes)]
    qs = [torch.rand(n, 2, device="cuda", generator=g) * 120 for n in (90, 7, 200)]
    a = tp.track_batch(clips, qs, coarse_iters=2)
    b = tp.track_batch(padded(clips), qs, coarse_iters=2, image_sizes=sizes_of(clips), num_frames=frames)
    assert set(a) == set(b)
    for k in a:
        _same(a[k], b[k], k)
    for k, v in a.items():
        if isinstance(v, torch.Tensor) and v.is_floating_point():
            assert torch.isfinite(v).all(), k


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["num_frames", "query_frames"])
def test_track_batch_mixed_sizes_against_track_calls(no_tf32, mode):
    """``track_batch`` over three sizes (one with 64x64 maps, the tensor path) against one ``track()`` per clip.  The
    arms take their coarse maps from different encoder calls (cuDNN may pick another algorithm for another frame count),
    and the iterated loop amplifies that rounding, so iteration 0 is held within 1e-4 of the maximum; the bitwise
    statements are the encoder and forward tests of this file."""
    import comet_pose_estimation_b200 as cb

    tp = _tracker()
    g = torch.Generator(device="cuda").manual_seed(6)
    frames = [8, 5, 6, 8] if mode == "num_frames" else [6, 6, 6, 6]
    sizes = [(512, 512), (384, 384), (480, 640), (384, 384)]
    clips = [torch.randn(s, 3, h, w, device="cuda", generator=g) for s, (h, w) in zip(frames, sizes)]
    qs = [torch.rand(n, 2, device="cuda", generator=g) * torch.tensor([w, h], device="cuda")
          for n, (h, w) in zip((200, 90, 150, 33), sizes)]
    qf = None
    if mode == "query_frames":
        qf = [torch.randint(0, s, (q.shape[0],), generator=torch.Generator().manual_seed(s + i))
              for i, (s, q) in enumerate(zip(frames, qs))]
    out = tp.track_batch(clips, qs, coarse_iters=2, query_frames=qf)
    assert out["image_sizes"].tolist() == [list(s) for s in sizes]
    parts = cb.split_batch(out)
    for b, (p, c, q) in enumerate(zip(parts, clips, qs)):
        one = tp.track(c[None], q[None], coarse_iters=2, query_frames=None if qf is None else qf[b])
        assert set(p) == set(one)
        for k, v in one.items():
            if isinstance(v, torch.Tensor):
                assert p[k].shape == v.shape, k
        assert rel_to_max(p["coarse_pred_track_list"][0].cpu(), one["coarse_pred_track_list"][0].cpu()) < 1e-4, b
        for k in ("refine_pred_track", "pred_score"):
            assert torch.isfinite(p[k]).all(), k
    for k, v in out.items():
        if isinstance(v, torch.Tensor) and v.dim() >= 3:
            assert torch.isfinite(v).all(), k


@pytest.mark.gpu
def test_graph_replays_for_a_new_mix_of_sizes(no_tf32):
    tp = _tracker()
    g = torch.Generator(device="cuda").manual_seed(7)
    make = lambda sizes: [torch.randn(6, 3, h, w, device="cuda", generator=g) for h, w in sizes]  # noqa: E731
    qs = [torch.rand(100, 2, device="cuda", generator=g) * 120 for _ in range(3)]
    former = tp.coarse_predictor.updateformer
    tp.track_batch(make([(256, 256), (128, 192), (256, 256)]), qs, coarse_iters=2, fine_tracking=False)
    captures = getattr(former, "_tc_captures", 0)
    out = tp.track_batch(make([(192, 160), (160, 128), (128, 128)]), qs, coarse_iters=2, fine_tracking=False)
    assert getattr(former, "_tc_captures", 0) == captures
    assert torch.isfinite(out["coarse_pred_track"]).all()


@pytest.mark.gpu
def test_smallest_size_runs(no_tf32):
    """``min_image_size()`` is a size ``track`` runs, alone and mixed with a larger size."""
    tp = _tracker()
    g = torch.Generator(device="cuda").manual_seed(10)
    m = tp.min_image_size()
    clips = [torch.randn(4, 3, m, m, device="cuda", generator=g), torch.randn(4, 3, m, m + 40, device="cuda", generator=g),
             torch.randn(3, 3, 256, 256, device="cuda", generator=g)]
    qs = [torch.rand(20, 2, device="cuda", generator=g) * m for _ in clips]
    one = tp.track(clips[0][None], qs[0][None], coarse_iters=1)
    out = tp.track_batch(clips, qs, coarse_iters=1)
    for v in (one["refine_pred_track"], out["refine_pred_track"], out["pred_score"]):
        assert torch.isfinite(v).all()
    with pytest.raises(AssertionError):
        tp.track_batch([clips[2], torch.randn(2, 3, m - 1, m, device="cuda")], qs[:2], coarse_iters=1)
