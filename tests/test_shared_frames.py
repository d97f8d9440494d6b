"""Clips that share frames of a video (``track_batch(clip_frames=...)``, the distinct-frame buffer, the item table and
source pools of any frame count in every layer below).  Contract: the call returns what ``track_batch`` returns for the
gathered clips ``[flat_frames[clip_frames[b]] for b in range(B)]``; each referenced frame is copied, encoded and prepared
once, and frames no clip references are never read.

Kernel-level results are held bitwise to the same kernels on explicitly gathered copies; loop-level results to the
float64 reference with the bars of test_full_size.py."""
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


def gather(videos, clip_frames):
    """The explicit copies the definition is stated on: clip b = flat_frames[clip_frames[b]]."""
    flat = [f for v in videos for f in v] if isinstance(videos, (list, tuple)) else list(videos)
    return [torch.stack([flat[int(t)] for t in c]) for c in clip_frames]


# ------------------------------------------------------------------------------------------------ CPU
def test_distinct_frame_buffer_and_item_tables():
    from comet_pose_estimation_b200.packed_frames import pack_referenced_frames
    from comet_pose_estimation_b200.utils import clip_items

    g = torch.Generator().manual_seed(0)
    videos = [torch.rand(6, 3, 8, 10, generator=g), torch.rand(5, 3, 12, 8, generator=g)]
    videos[0][4] = float("nan")                                     # frames 4 and 9 are referenced by no clip
    videos[1][3] = float("nan")
    clips = [[5, 3, 3, 1], [7, 6, 10], [0, 1, 2, 3, 5], [10, 8, 7]]  # repeats, shared frames, descending, two sizes
    packed, ids = pack_referenced_frames(videos, clips)
    used = sorted({t for c in clips for t in c})
    assert packed.num_frames == len(used) == 9
    assert torch.isfinite(packed.data).all()                          # unreferenced frames are not in the buffer
    frame = lambda t: videos[0][t] if t < 6 else videos[1][t - 6]  # noqa: E731
    for c, row in zip(clips, ids):
        for t, f in zip(c, row):
            assert torch.equal(packed.frames(f, 1)[0], frame(t))
    assert ids[0][1] == ids[0][2] and ids[0][1] == ids[2][3]          # one packed frame per source frame
    assert [hw for hw, _ in packed.groups] == [(8, 10), (12, 8)]
    assert len(packed.groups[0][1]) == 2                              # runs 0..3 and 5 of video 0

    group_of = [0, 1, 0, 1]
    qf = [[0, 2, 2], [1], [0, 4], [0, 0]]
    items, pos, table = clip_items(ids, qf, group_of)
    assert [(b, q, ns) for b, q, ns in items] == [(0, 0, [0]), (0, 2, [1, 2]), (2, 0, [0]), (2, 4, [1]),
                                                  (1, 1, [0]), (3, 0, [0, 1])]
    assert pos.shape == table.shape == (6, 5) and pos.dtype == table.dtype == torch.int64
    assert pos[1].tolist() == [2, 1, 0, 3, 4]                         # the query-position swap
    assert pos[3].tolist() == [4, 1, 2, 3, 0]
    assert pos[4].tolist() == [1, 0, 2, 3, 4]                         # positions 3.. of a 3-frame clip are padding
    for i, (b, _, _) in enumerate(items):
        for s in range(5):
            p = int(pos[i, s])
            assert table[i, s] == ids[b][min(p, len(ids[b]) - 1)]
    assert table[1].tolist() == [ids[0][2], ids[0][1], ids[0][0], ids[0][3], ids[0][3]]


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
            m = fmaps.mean(dim=(2, 3, 4)) + fmaps.shape[-1] * 1e-3
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


def _bad_calls():
    g = torch.Generator().manual_seed(0)
    video = torch.rand(6, 3, 64, 64, generator=g)
    other = torch.rand(3, 3, 72, 64, generator=g)
    qs = [torch.zeros(3, 2), torch.zeros(2, 2)]
    ok = [[0, 1, 2], [3, 4]]
    return [(video, qs, dict(clip_frames=[[0.0, 1.0, 2.0], [3, 4]])),                 # not integers
            (video, qs, dict(clip_frames=[torch.tensor([0, 1.5]), torch.tensor([3, 4])])),
            (video, qs, dict(clip_frames=[[0, 1, 6], [3, 4]])),                       # past the last frame
            (video, qs, dict(clip_frames=[[0, -1], [3, 4]])),                         # negative
            (video, qs, dict(clip_frames=[[0, 1], []])),                              # empty clip
            ([video, other], qs, dict(clip_frames=[[0, 1, 6], [7, 8]])),              # a clip mixing sizes
            (video, qs, dict(clip_frames=[[0, 1], [2, 3], [4, 5]])),                  # three clips, two query lists
            (video, qs, dict(clip_frames=ok, num_frames=[3, 3])),                     # num_frames disagrees
            ([video, other], qs, dict(clip_frames=[[0], [6]], image_sizes=[[64, 64], [64, 72]])),
            ([video, torch.rand(2, 3, 63, 64, generator=g)], qs, dict(clip_frames=[[0], [6, 7]]))]   # below the floor


@pytest.mark.parametrize("k", range(10))
def test_invalid_clip_frames_are_refused(k):
    tp = _stub_tracker()
    images, qs, kw = _bad_calls()[k]
    with pytest.raises(AssertionError):
        tp.track_batch(images, qs, fine_tracking=False, **kw)


def test_cpu_forward_with_source_pool_equals_gathered_maps():
    """The CPU definition of the layer: a pool of S_src != S source frames read through the table == the forward on the
    gathered maps, for one pool and for per-group pools of different sizes and frame counts."""
    tp = _stub_tracker()
    m = tp.coarse_predictor
    g = torch.Generator().manual_seed(1)
    pool = torch.rand(2, 7, 4, 8, 8, generator=g)                     # 14 source frames, items of 5 positions
    fi = torch.tensor([[3, 3, 9, 1, 0], [13, 12, 11, 10, 9], [13, 12, 11, 10, 9], [4, 5, 6, 7, 7]])
    q = torch.rand(4, 3, 2, generator=g) * 7
    kw = dict(iters=2, return_feat=True, TRACKorPOSE=False, num_tracks=[3, 1, 2, 3], num_frames=[5, 5, 4, 2])
    with torch.no_grad():
        got = m(query_points=q, fmaps=pool, frame_index=fi, **kw)
        want = m(query_points=q, fmaps=pool.flatten(0, 1)[fi], **kw)
        assert all(torch.equal(a, b) for a, b in zip(got[0], want[0])) and torch.equal(got[1], want[1])
        other = torch.rand(1, 3, 4, 6, 10, generator=g)              # a second size group with 3 source frames
        fi2 = torch.cat([fi, torch.tensor([[2, 0, 0, 1, 2]])])
        q2 = torch.cat([q, torch.rand(1, 3, 2, generator=g) * 5])
        kw2 = dict(kw, num_tracks=[3, 1, 2, 3, 2], num_frames=[5, 5, 4, 2, 5])
        got = m(query_points=q2, fmaps=[pool, other], frame_index=fi2, group_items=[4, 1], **kw2)
        for r0, r1, f in ((0, 4, pool), (4, 5, other)):
            want = m(query_points=q2[r0:r1], fmaps=f.flatten(0, 1)[fi2[r0:r1]], iters=2, return_feat=True,
                     TRACKorPOSE=False, num_tracks=kw2["num_tracks"][r0:r1], num_frames=kw2["num_frames"][r0:r1])
            assert all(torch.equal(a[r0:r1], b) for a, b in zip(got[0], want[0])) and torch.equal(got[1][r0:r1], want[1])


def _cpu_batch():
    g = torch.Generator().manual_seed(2)
    videos = [torch.rand(7, 3, 64, 80, generator=g), torch.rand(4, 3, 72, 64, generator=g)]
    clips = [torch.tensor([0, 1, 2, 3]), [2, 3, 4, 5, 6], [6, 5, 5, 2], [8, 7, 10]]
    qs = [torch.rand(n, 2, generator=g) * 60 for n in (5, 2, 4, 3)]
    qf = [torch.tensor([0, 3, 3, 1, 0]), torch.tensor([4, 1]), torch.tensor([0, 0, 2, 0]), torch.tensor([1, 0, 2])]
    return videos, clips, qs, qf


@pytest.mark.parametrize("mode", ["one_size", "two_sizes", "query_frames"])
def test_cpu_clip_frames_equal_gathered_clips(mode):
    """The definition on the CPU: the call equals ``track_batch`` on the gathered clips, with the same keys."""
    tp = _stub_tracker()
    videos, clips, qs, qf = _cpu_batch()
    if mode == "one_size":
        videos, clips, qs = videos[0], clips[:3], qs[:3]
    kw = dict(query_frames=qf) if mode == "query_frames" else {}
    with torch.no_grad():
        got = tp.track_batch(videos, qs, fine_tracking=False, clip_frames=clips, **kw)
        want = tp.track_batch(gather(videos, clips), qs, fine_tracking=False, **kw)
    assert set(got) == set(want)
    assert ("image_sizes" in got) == (mode != "one_size") and "num_frames" in got
    for k, v in want.items():
        if isinstance(v, list):
            assert all(torch.allclose(a, b, rtol=1e-6, atol=1e-6) for a, b in zip(got[k], v)), k
        elif isinstance(v, torch.Tensor):
            assert got[k].shape == v.shape and got[k].dtype == v.dtype, k
            assert torch.allclose(got[k].double(), v.double(), rtol=1e-6, atol=1e-6), k


def test_cpu_split_batch_on_clip_frames_result():
    import comet_pose_estimation_b200 as cb

    tp = _stub_tracker()
    videos, clips, qs, qf = _cpu_batch()
    with torch.no_grad():
        out = tp.track_batch(videos, qs, fine_tracking=False, clip_frames=clips, query_frames=qf)
        parts = cb.split_batch(out)
        assert len(parts) == 4
        for b, (c, q, t) in enumerate(zip(gather(videos, clips), qs, qf)):
            one = tp.track(c[None], q[None], fine_tracking=False, query_frames=t)
            assert set(parts[b]) == set(one)
            for k in ("coarse_pred_track", "vis", "pred_score", "refine_pred_track"):
                assert parts[b][k].shape == one[k].shape, k
                assert torch.allclose(parts[b][k], one[k], rtol=1e-6, atol=1e-6), (k, b)
            assert torch.equal(parts[b]["query_frames"], one["query_frames"])


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture
def no_tf32():
    a, b = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = a, b


# 2 x 7 = 14 source frames, items of S = 5 positions: BS_src is no multiple of S; a row with repeats, two identical rows,
# a descending row; frames 2 and 8 are referenced by no row
POOL_B, POOL_S, S = 2, 7, 5
TABLE = torch.tensor([[3, 3, 9, 1, 0], [13, 12, 11, 10, 9], [13, 12, 11, 10, 9], [4, 5, 6, 7, 7], [0, 0, 0, 0, 0]])
UNREFERENCED = (2, 8)


def _nan_unreferenced(x):
    flat = x.flatten(0, 1)
    for f in UNREFERENCED:
        flat[f] = float("nan")
    return x


@pytest.mark.gpu
@pytest.mark.parametrize("tensor_path", [True, False])
@pytest.mark.parametrize("autocast", [False, True])
@pytest.mark.parametrize("counts", [False, True])
def test_tokens_from_source_pool(no_tf32, tensor_path, autocast, counts):
    import comet_pose_estimation_b200 as cb

    if tensor_path and not cb._lib.lib.comet_has_tensor_path():
        pytest.skip("no sm_100 tensor path on this device")
    g = torch.Generator(device="cuda").manual_seed(5)
    L, r = 4, 3
    fi = TABLE.cuda()
    Bi = fi.shape[0]
    nt, nf = ([300, 137, 1, 64, 200], [5, 5, 3, 4, 1]) if counts else (None, None)
    N = 300
    fmaps = _nan_unreferenced(torch.randn(POOL_B, POOL_S, 128, 64, 64, device="cuda", generator=g))
    feats = torch.randn(Bi, S, N, 128, device="cuda", generator=g)
    coords = torch.rand(Bi, S, N, 2, device="cuda", generator=g) * 70 - 3
    tdim = max(cb.transformer_dim(L, r, 128, False), (2 * 128 + 2 + L * (2 * r + 1) ** 2 + 3) // 4 * 4)
    prev = cb._lib.set_option(cb._lib.OPT_TENSOR_PATH, tensor_path)
    try:
        ctx = torch.autocast("cuda", dtype=torch.bfloat16) if autocast else contextlib.nullcontext()
        with ctx, torch.no_grad():
            blk = cb.CorrBlock(fmaps, num_levels=L, radius=r)
            assert (blk._pyr.split is not None) == tensor_path
            got = cb.TrackTokenizer(blk, coords[:, 0], tdim, num_tracks=nt, num_frames=nf,
                                    frame_index=fi).tokens(coords, feats).clone()
            copy = cb.CorrBlock(fmaps.flatten(0, 1)[fi], num_levels=L, radius=r)
            want = cb.TrackTokenizer(copy, coords[:, 0], tdim, num_tracks=nt, num_frames=nf).tokens(coords, feats)
            assert torch.equal(got, want)
            assert torch.isfinite(got).all()
    finally:
        cb._lib.set_option(cb._lib.OPT_TENSOR_PATH, prev)
    if tensor_path:
        assert cb._lib.lib.comet_tc_status() == 0


@pytest.mark.gpu
@pytest.mark.parametrize("counts", [False, True])
def test_patch_encoder_from_source_pool(no_tf32, counts):
    """The indexed and the packed patch encoder reading a pool of 14 frames through 5-position rows == the varlen
    encoder on the gathered images."""
    import comet_pose_estimation_b200 as cb

    fnet = load_seeded(cb.ShallowEncoder(input_dim=3).eval(), 3).cuda()
    g = torch.Generator(device="cuda").manual_seed(2)
    H, W = 96, 80
    fi = TABLE.cuda()
    tracks = [2, 1, 3, 1, 2]
    images = _nan_unreferenced(torch.randn(POOL_B, POOL_S, 3, H, W, device="cuda", generator=g))
    tl = (torch.rand(len(tracks), S, max(tracks), 2, device="cuda", generator=g) * 90 - 10).floor().int()
    seq = torch.tensor([i for i, n in enumerate(tracks) for _ in range(n)], device="cuda")
    loc = torch.tensor([j for n in tracks for j in range(n)], device="cuda")
    nf = torch.tensor([5, 5, 3, 4, 1], dtype=torch.int32, device="cuda") if counts else None
    packed = cb.PackedFrames([images.flatten(0, 1)])
    with torch.no_grad():
        got, _ = fnet.encode_packed_patches_of(images, tl[seq, :, loc], seq, num_frames=nf, frame_index=fi)
        via_packed, _ = fnet.encode_packed_frames_patches_of(packed, tl[seq, :, loc], seq, num_frames=nf, frame_index=fi)
        want, _ = fnet.encode_packed_patches_of(images.flatten(0, 1)[fi], tl[seq, :, loc], seq, num_frames=nf)
    assert torch.equal(got, want) and torch.equal(via_packed, want)
    assert torch.isfinite(got).all()


def _coarse_model():
    import comet_pose_estimation_b200 as cb

    return load_seeded(cb.BaseTrackerPredictor(cfg=cfg(), **cases.FULL_COARSE_CTOR).eval(), cases.FULL_SEEDS["coarse"]).cuda()


def _fine_models():
    import comet_pose_estimation_b200 as cb

    fnet = load_seeded(cb.ShallowEncoder(input_dim=3).eval(), cases.FULL_SEEDS["fnet"]).cuda()
    ftr = load_seeded(cb.BaseTrackerPredictor(cfg=cfg(), **cases.FULL_FINE_CTOR).eval(), cases.FULL_SEEDS["fine"]).cuda()
    return fnet.to(memory_format=torch.channels_last), ftr


@pytest.mark.gpu
@pytest.mark.parametrize("side", [64, 48])                          # tensor path / SIMT path
@pytest.mark.parametrize("autocast", [False, True])
def test_coarse_forward_from_source_pool(no_tf32, side, autocast):
    g = torch.Generator(device="cuda").manual_seed(3)
    m = _coarse_model()
    fi = TABLE.cuda()
    counts, frames = [300, 37, 512, 64, 1], [5, 5, 3, 4, 2]
    fmaps = _nan_unreferenced(torch.randn(POOL_B, POOL_S, 128, side, side, device="cuda", generator=g))
    q = torch.rand(len(counts), max(counts), 2, device="cuda", generator=g) * side * 8
    kw = dict(iters=3, return_feat=True, TRACKorPOSE=False, down_ratio=2, num_tracks=counts, num_frames=frames)
    ctx = torch.autocast("cuda", dtype=torch.bfloat16) if autocast else contextlib.nullcontext()
    with ctx, torch.no_grad():
        got = m(query_points=q, fmaps=fmaps, frame_index=fi, **kw)
        want = m(query_points=q, fmaps=fmaps.flatten(0, 1)[fi], **kw)
    for i, (a, b) in enumerate(zip(got[0], want[0])):
        assert torch.equal(a, b), i
    for a, b in zip(got[1:], want[1:]):
        assert (a is None and b is None) or torch.equal(a, b)
    assert torch.isfinite(got[0][-1]).all()


@pytest.mark.gpu
def test_refine_from_source_pool(no_tf32):
    import comet_pose_estimation_b200 as cb

    fnet, ftr = _fine_models()
    g = torch.Generator(device="cuda").manual_seed(13)
    fi = TABLE.cuda()
    counts, frames = [40, 7, 64, 1, 30], [5, 5, 3, 4, 2]
    images = _nan_unreferenced(torch.rand(POOL_B, POOL_S, 3, 128, 128, device="cuda", generator=g))
    coarse = torch.rand(len(counts), S, max(counts), 2, device="cuda", generator=g) * 127
    kw = dict(compute_score=True, num_tracks=counts, num_frames=frames)
    with torch.no_grad():
        got = cb.refine_track(images, fnet, ftr, coarse, frame_index=fi, **kw)
        packed = cb.refine_track(cb.PackedFrames([images.flatten(0, 1)]), fnet, ftr, coarse, frame_index=fi, **kw)
        want = cb.refine_track(images.flatten(0, 1)[fi], fnet, ftr, coarse, **kw)
    for a in (got, packed):
        assert torch.equal(a[0], want[0]) and torch.equal(a[1], want[1])
    assert torch.isfinite(got[0]).all() and torch.isfinite(got[1]).all()


def _window_table(S_golden):
    """Clips [0,16), [4,20), [8,24) of a 24-frame video whose frames 4..19 are the golden sequence."""
    return torch.stack([torch.arange(s, s + S_golden) for s in (0, 4, 8)])


@pytest.mark.gpu
def test_golden_coarse_case_as_middle_window(golden, no_tf32):
    g = golden("tracker_full")
    m = _coarse_model()
    fmaps, q = cases.tracker_case(**cases.FULL_COARSE_CASE)
    fmaps, q = torch.from_numpy(fmaps).cuda(), torch.from_numpy(q).cuda()
    S_g, N = fmaps.shape[1], q.shape[1]
    H, W = fmaps.shape[-2:]
    scale = cases.FULL_COARSE_CASE["down_ratio"] * 4
    gen = torch.Generator(device="cuda").manual_seed(9)
    video = torch.randn((1, S_g + 8) + tuple(fmaps.shape[2:]), device="cuda", generator=gen)
    video[0, 4:4 + S_g] = fmaps[0]
    counts = [300, N, 137]
    qp = torch.rand(3, N, 2, device="cuda", generator=gen) * torch.tensor([W, H], device="cuda") * scale * 0.9
    qp[1] = q[0]
    with torch.no_grad():
        preds, vis, _, _, _ = m(query_points=qp, fmaps=video, iters=cases.FULL_COARSE_ITERS, return_feat=True,
                                down_ratio=cases.FULL_COARSE_CASE["down_ratio"], TRACKorPOSE=False, num_tracks=counts,
                                frame_index=_window_table(S_g).cuda())
    for i in range(cases.FULL_COARSE_ITERS):
        assert rel_to_max(preds[i][1:2].cpu().numpy(), g[f"pred64_{i}"]) <= bar(g[f"pred32_{i}"], g[f"pred64_{i}"]), i
    assert rel_to_max(vis[1:2].cpu().numpy(), g["vis64"]) <= bar(g["vis32"], g["vis64"])
    assert all(torch.isfinite(p).all() for p in preds)


@pytest.mark.gpu
def test_golden_refine_case_as_middle_window(golden, no_tf32):
    import comet_pose_estimation_b200 as cb

    r = golden("refine_full")
    fnet, ftr = _fine_models()
    images, _ = cases.refine_case(**cases.FULL_REFINE_CASE)
    images = torch.from_numpy(images).cuda()
    coarse = torch.from_numpy(r["coarse_pred"]).cuda()
    S_g, N = coarse.shape[1], coarse.shape[2]
    g = torch.Generator(device="cuda").manual_seed(4)
    video = torch.rand((1, S_g + 8) + tuple(images.shape[2:]), device="cuda", generator=g)
    video[0, 4:4 + S_g] = images[0]
    counts = [137, N, 300]
    batch_c = torch.zeros(3, S_g, N, 2, device="cuda")
    batch_c[1] = coarse[0]
    for i in (0, 2):
        perm = torch.randperm(N, generator=torch.Generator().manual_seed(i))[:counts[i]].cuda()
        batch_c[i, :, :counts[i]] = coarse[0, :, perm] + 3.0
    with torch.no_grad():
        refined, score = cb.refine_track(video, fnet, ftr, batch_c, compute_score=True, num_tracks=counts,
                                         frame_index=_window_table(S_g).cuda())
    inv = cb.inverted_score(score[1:2])
    for k, got in (("refined", refined[1:2]), ("score", score[1:2]), ("inverted", inv)):
        assert rel_to_max(got.cpu().numpy(), r[k + "64"]) <= bar(r[k + "32"], r[k + "64"]), k
    assert torch.isfinite(refined).all() and torch.isfinite(score).all()


def _tracker():
    import comet_pose_estimation_b200 as cb

    torch.manual_seed(0)
    return cb.TrackerPredictor().eval().cuda()


def _per_frame_encoder(tp):
    """Make the coarse encoder batch-independent: every frame is encoded by a call of its own (cuDNN then sees one
    batch size in both arms of a comparison)."""
    enc = tp._encode_flat
    tp._encode_flat = lambda x: torch.cat([enc(x[i:i + 1]) for i in range(x.shape[0])])


def _same(a, b, k):
    if isinstance(a, list):
        assert len(a) == len(b) and all(torch.equal(x, y) for x, y in zip(a, b)), k
    elif a is None:
        assert b is None, k
    else:
        assert a.shape == b.shape and torch.equal(a, b), k


def _video_batch(g, T=24, side=256):
    video = torch.randn(T, 3, side, side, device="cuda", generator=g)
    clips = [list(range(0, 16)), list(range(8, 24)), [5, 3, 3, 1, 20, 19, 18, 0, 7], list(range(23, 11, -1))]
    qs = [torch.rand(n, 2, device="cuda", generator=g) * (side - 10) for n in (120, 33, 64, 90)]
    return video, clips, qs


@pytest.mark.gpu
@pytest.mark.parametrize("query_frames", [False, True])
def test_clip_frames_bit_identical_to_gathered_clips_with_a_per_frame_encoder(no_tf32, query_frames):
    tp = _tracker()
    _per_frame_encoder(tp)
    g = torch.Generator(device="cuda").manual_seed(11)
    video, clips, qs = _video_batch(g)
    kw = {}
    if query_frames:
        kw["query_frames"] = [torch.randint(0, len(c), (q.shape[0],), generator=torch.Generator().manual_seed(b))
                              for b, (c, q) in enumerate(zip(clips, qs))]
    got = tp.track_batch(video, qs, coarse_iters=3, clip_frames=clips, **kw)
    want = tp.track_batch(gather(video, clips), qs, coarse_iters=3, **kw)
    assert set(got) == set(want)
    for k in want:
        _same(got[k], want[k], k)
    assert torch.isfinite(got["refine_pred_track"]).all()


@pytest.mark.gpu
def test_clip_frames_against_gathered_clips_at_iteration_0(no_tf32):
    """With the real encoder the two arms call cuDNN with different frame counts, and the iterated loop amplifies that
    rounding: iteration 0 is held within 1e-4 of the maximum."""
    tp = _tracker()
    g = torch.Generator(device="cuda").manual_seed(12)
    video, clips, qs = _video_batch(g)
    got = tp.track_batch(video, qs, coarse_iters=2, clip_frames=clips)
    want = tp.track_batch(gather(video, clips), qs, coarse_iters=2)
    assert set(got) == set(want)
    assert rel_to_max(got["coarse_pred_track_list"][0].cpu(), want["coarse_pred_track_list"][0].cpu()) < 1e-4
    assert torch.isfinite(got["refine_pred_track"]).all()


@pytest.mark.gpu
def test_windows_are_encoded_once(no_tf32):
    tp = _tracker()
    seen = []
    h = tp.coarse_fnet.register_forward_hook(lambda mod, inp, out: seen.append(inp[0].shape[0]))
    g = torch.Generator(device="cuda").manual_seed(1)
    video = torch.randn(40, 3, 256, 256, device="cuda", generator=g)
    clips = [list(range(s, s + 16)) for s in (0, 8, 16, 24)]
    qs = [torch.rand(40, 2, device="cuda", generator=g) * 240 for _ in clips]
    try:
        out = tp.track_batch(video, qs, coarse_iters=1, fine_tracking=False, clip_frames=clips)
    finally:
        h.remove()
    assert seen == [40]
    assert out["coarse_pred_track"].shape == (4, 16, 40, 2)


@pytest.mark.gpu
def test_unreferenced_frames_are_not_read(no_tf32):
    tp = _tracker()
    g = torch.Generator(device="cuda").manual_seed(2)
    video = torch.randn(30, 3, 256, 256, device="cuda", generator=g)
    clips = [list(range(0, 10)), [12, 14, 16, 18, 29], [29, 0, 14]]
    unused = sorted(set(range(30)) - {t for c in clips for t in c})
    qs = [torch.rand(n, 2, device="cuda", generator=g) * 240 for n in (50, 20, 7)]
    a, b = video.clone(), video.clone()
    a[unused] = float("nan")
    b[unused] = 0.0
    got = tp.track_batch(a, qs, coarse_iters=2, clip_frames=clips)
    want = tp.track_batch(b, qs, coarse_iters=2, clip_frames=clips)
    for k in want:
        _same(got[k], want[k], k)
    assert torch.isfinite(got["refine_pred_track"]).all() and torch.isfinite(got["pred_score"]).all()


@pytest.mark.gpu
def test_composition_of_counts_lengths_query_frames_and_two_sizes(no_tf32):
    """Ragged track counts, clips of 9-16 frames, query frames and two videos of 512x512 (tensor path) and 384x384 (SIMT)
    in one call == ``track_batch`` on the gathered clips, bit for bit with a per-frame encoder."""
    import comet_pose_estimation_b200 as cb

    tp = _tracker()
    _per_frame_encoder(tp)
    g = torch.Generator(device="cuda").manual_seed(3)
    videos = [torch.randn(20, 3, 512, 512, device="cuda", generator=g), torch.randn(18, 3, 384, 384, device="cuda", generator=g)]
    clips = [list(range(0, 16)), list(range(24, 33)), list(range(4, 16)), list(range(37, 21, -1)), list(range(8, 20))]
    qs = [torch.rand(n, 2, device="cuda", generator=g) * 370 for n in (200, 31, 128, 77, 5)]
    qf = [torch.randint(0, len(c), (q.shape[0],), generator=torch.Generator().manual_seed(b))
          for b, (c, q) in enumerate(zip(clips, qs))]
    got = tp.track_batch(videos, qs, coarse_iters=2, clip_frames=clips, query_frames=qf)
    want = tp.track_batch(gather(videos, clips), qs, coarse_iters=2, query_frames=qf)
    assert got["image_sizes"].tolist() == [[512, 512], [384, 384], [512, 512], [384, 384], [512, 512]]
    assert set(got) == set(want)
    for k in want:
        _same(got[k], want[k], k)
    for b, p in enumerate(cb.split_batch(got)):
        assert p["coarse_pred_track"].shape == (1, len(clips[b]), qs[b].shape[0], 2)
        assert torch.isfinite(p["refine_pred_track"]).all()


@pytest.mark.gpu
def test_graph_replays_for_a_new_clip_table(no_tf32):
    tp = _tracker()
    g = torch.Generator(device="cuda").manual_seed(7)
    video = torch.randn(30, 3, 256, 256, device="cuda", generator=g)
    former = tp.coarse_predictor.updateformer
    first = [list(range(0, 8)), list(range(4, 12)), list(range(20, 28))]
    second = [list(range(29, 21, -1)), [0, 0, 1, 1, 2, 2, 3, 3], list(range(10, 18))]     # the same (B', N_cap, S_max)
    tp.track_batch(video, [torch.rand(n, 2, device="cuda", generator=g) * 240 for n in (100, 60, 90)], coarse_iters=2,
                   fine_tracking=False, clip_frames=first)
    captures = getattr(former, "_tc_captures", 0)
    out = tp.track_batch(video, [torch.rand(n, 2, device="cuda", generator=g) * 240 for n in (70, 100, 30)],
                         coarse_iters=2, fine_tracking=False, clip_frames=second)
    assert getattr(former, "_tc_captures", 0) == captures
    assert torch.isfinite(out["coarse_pred_track"]).all()
