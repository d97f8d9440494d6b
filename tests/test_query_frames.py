"""Tracks whose query points lie on any frame (``query_frames=`` on ``track`` / ``track_batch`` and the ``frame_index``
table of every layer below them).  Contract: track n of sequence b with query frame q gets what ``track_batch`` returns
for it on one item -- sequence b's images with frames 0 and q swapped, the tracks of sequence b whose query frame is q,
S_b frames -- with every per-frame output swapped back.  The frames are encoded once; items read them through the table.

Kernel-level results are held bitwise to the same kernels on explicitly gathered copies (every item reads the same values
in the same order as its copy); loop-level results to the float64 reference with the bars of test_full_size.py."""
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
    """Frames 0 and q of ``x`` swapped along ``dim`` (VGGSfM's switch_tensor_order)."""
    order = list(range(x.shape[dim]))
    order[0], order[q] = q, 0
    return x.index_select(dim, torch.tensor(order, device=x.device))


# ------------------------------------------------------------------------------------------------ CPU
def test_items_and_frame_index_table():
    from comet_pose_estimation_b200.utils import query_frame_items

    frames, S = [6, 3, 5], 6
    qf = [[0, 2, 2, 5], [1, 1], [0, 4, 0]]
    items, fi = query_frame_items(qf, frames, S)
    assert [(b, q, ns) for b, q, ns in items] == [(0, 0, [0]), (0, 2, [1, 2]), (0, 5, [3]), (1, 1, [0, 1]),
                                                  (2, 0, [0, 2]), (2, 4, [1])]
    assert fi.shape == (6, S) and fi.dtype == torch.int64
    assert fi[0].tolist() == [0, 1, 2, 3, 4, 5]                        # q = 0: identity
    assert fi[1].tolist() == [2, 1, 0, 3, 4, 5]                        # one swap per item
    assert fi[2].tolist() == [5, 1, 2, 3, 4, 0]
    assert fi[3].tolist() == [7, 6, 8, 9, 10, 11]                      # positions 3..5 padded: identity
    assert fi[5].tolist() == [16, 13, 14, 15, 12, 17]                  # position 5 padded: identity
    # the items of one sequence share its source frames, in different orders
    assert sorted(fi[0].tolist()) == sorted(fi[1].tolist()) == sorted(fi[2].tolist())
    assert sorted(fi[4].tolist()) == sorted(fi[5].tolist()) == list(range(12, 18))


def _stub_tracker():
    """A TrackerPredictor whose coarse predictor is the real ``BaseTrackerPredictor.forward`` for the frame-table
    handling (on the CPU it gathers the maps and calls itself again) around a cheap frame-order-dependent computation."""
    import comet_pose_estimation_b200 as cb

    class Stub(cb.BaseTrackerPredictor):
        def forward(self, query_points, fmaps=None, iters=4, return_feat=False, down_ratio=1, is_train=False,
                    track_feats=None, TRACKorPOSE=True, ind=0, num_tracks=None, num_frames=None, frame_index=None):
            if frame_index is not None:
                return super().forward(query_points, fmaps, iters, return_feat, down_ratio, is_train, track_feats,
                                       TRACKorPOSE, ind, num_tracks, num_frames, frame_index)
            B, S = fmaps.shape[:2]
            N = query_points.shape[1]
            m = fmaps.mean(dim=(2, 3, 4))                                      # (B, S)
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


def _bad_query_frames():
    return [torch.tensor([[0, -1, 0], [0, 0, 0]]),                   # negative
            torch.tensor([[0, 1, 0], [0, 3, 0]]),                    # >= S_b (sequence 1 has 3 frames)
            [torch.tensor([0, 1, 0])],                               # one list for two sequences
            [torch.tensor([0, 1]), torch.tensor([0, 1, 2])],         # lengths disagree with the tracks
            torch.tensor([[0.0, 1.0, 0.0], [0.0, 0.0, 0.0]])]        # not integers


@pytest.mark.parametrize("k", range(5))
def test_invalid_query_frames_are_refused(k):
    tp = _stub_tracker()
    images = torch.zeros(2, 4, 3, 8, 8)
    qs = [torch.zeros(3, 2), torch.zeros(3, 2)]
    with pytest.raises(AssertionError):
        tp.track_batch(images, qs, num_frames=[4, 3], fine_tracking=False, query_frames=_bad_query_frames()[k])
    with pytest.raises(AssertionError):
        tp.track(images[:1], qs[0][None], fine_tracking=False, query_frames=torch.tensor([0, 4, 0]))


def test_cpu_forward_equals_swapped_items_scattered_back():
    """The CPU definition: every (sequence, query frame) item is the call on explicitly swapped images, scattered back."""
    import comet_pose_estimation_b200 as cb

    tp = _stub_tracker()
    g = torch.Generator().manual_seed(1)
    frames, S = [6, 3, 5], 6
    clips = [torch.rand(s, 3, 8, 8, generator=g) for s in frames]
    qs = [torch.rand(n, 2, generator=g) * 8 for n in (5, 2, 4)]
    qf = [torch.tensor([0, 3, 3, 5, 0]), torch.tensor([2, 1]), torch.tensor([4, 0, 4, 1])]
    with torch.no_grad():
        out = tp.track_batch(clips, qs, fine_tracking=False, query_frames=qf)
        assert out["query_frames"].shape == (3, 5) and out["query_frames"].dtype == torch.int64
        for b, (c, q, t) in enumerate(zip(clips, qs, qf)):
            n, s = q.shape[0], c.shape[0]
            assert out["query_frames"][b, :n].tolist() == t.tolist()
            for qq in sorted(set(t.tolist())):
                sel = torch.nonzero(t == qq)[:, 0]
                one = tp.track_batch(swap(c[None], qq), q[None, sel], fine_tracking=False)
                for k in ("coarse_pred_track", "vis", "pred_score", "refine_pred_track"):
                    want = swap(one[k], qq)[0]
                    assert torch.allclose(out[k][b, :s, sel], want, rtol=1e-6, atol=1e-6), (k, b, qq)
                for i, lvl in enumerate(out["coarse_pred_track_list"]):
                    assert torch.allclose(lvl[b, :s, sel], swap(one["coarse_pred_track_list"][i], qq)[0], rtol=1e-6,
                                          atol=1e-6)
            for k in ("coarse_pred_track", "vis", "pred_score"):
                assert torch.count_nonzero(out[k][b, s:]) == 0 and torch.count_nonzero(out[k][b, :, n:]) == 0
        parts = cb.split_batch(out)
        one = tp.track(clips[1][None], qs[1][None], fine_tracking=False, query_frames=qf[1])
        assert set(one) == set(parts[1])
        for k, v in one.items():
            if isinstance(v, torch.Tensor):
                assert torch.equal(v, parts[1][k]), k


def test_query_frame_zero_tracks_are_untouched_by_the_swap():
    """Scattering back is an exact inverse: tracks with t_n = 0 equal the call with those tracks alone."""
    tp = _stub_tracker()
    g = torch.Generator().manual_seed(2)
    images = torch.rand(2, 5, 3, 8, 8, generator=g)
    qp = torch.rand(2, 4, 2, generator=g) * 8
    qf = torch.tensor([[0, 2, 0, 4], [3, 0, 0, 1]])
    with torch.no_grad():
        out = tp.track_batch(images, qp, fine_tracking=False, query_frames=qf)
        for b in range(2):
            sel = torch.nonzero(qf[b] == 0)[:, 0]
            one = tp.track_batch(images[b:b + 1], qp[b:b + 1, sel], fine_tracking=False)
            for k in ("coarse_pred_track", "vis", "pred_score"):
                assert torch.equal(out[k][b, :, sel], one[k][0]), (k, b)


def test_split_batch_cuts_query_frames():
    import comet_pose_estimation_b200 as cb

    B, S, N = 3, 5, 7
    counts, frames = [7, 1, 4], [5, 2, 1]
    t = lambda *s: torch.randn(*s)  # noqa: E731
    qf = torch.randint(0, 5, (B, N))
    out = {"coarse_pred_track_list": [t(B, S, N, 2) for _ in range(4)], "coarse_pred_track": t(B, S, N, 2),
           "vis": t(B, S, N), "conf": None, "refine_pred_track": t(B, S, N, 2), "track_score": t(B, S, N),
           "pred_score": t(B, S, N), "num_tracks": torch.tensor(counts), "num_frames": torch.tensor(frames),
           "query_frames": qf}
    for p, n, s, b in zip(cb.split_batch(out), counts, frames, range(B)):
        assert set(p) == set(out) - {"num_tracks", "num_frames"}
        assert p["query_frames"].shape == (1, n) and torch.equal(p["query_frames"][0], qf[b, :n])
        assert p["coarse_pred_track"].shape == (1, s, n, 2) and p["vis"].shape == (1, s, n)


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture
def no_tf32():
    a, b = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = a, b


def _table(frames, qs, S):
    from comet_pose_estimation_b200.utils import query_frame_items

    items, fi = query_frame_items(qs, frames, S)
    return [b for b, _, _ in items], fi


@pytest.mark.gpu
@pytest.mark.parametrize("tensor_path", [True, False])
@pytest.mark.parametrize("autocast", [False, True])
def test_coarse_tokens_with_frame_table(no_tf32, tensor_path, autocast):
    """Tensor and SIMT token kernels reading the source pyramid through the table == the same kernels on the gathered
    maps, with track and frame counts mixed in; padded rows are 0."""
    import comet_pose_estimation_b200 as cb

    if tensor_path and not cb._lib.lib.comet_has_tensor_path():
        pytest.skip("no sm_100 tensor path on this device")
    g = torch.Generator(device="cuda").manual_seed(5)
    S, L, r = 5, 4, 3
    seq, fi = _table([5, 3], [[0, 2, 4, 2], [1, 0]], S)          # items (0,0) (0,2) (0,4) (1,0) (1,1)
    counts, frames = [300, 137, 1, 64, 200], [5, 5, 5, 3, 3]
    Bi, N = len(counts), max(counts)
    fmaps = torch.randn(2, S, 128, 64, 64, device="cuda", generator=g)
    fmaps[1, 3:] = 0.0                                             # what the encoder leaves in padded frames
    feats = torch.randn(Bi, S, N, 128, device="cuda", generator=g)
    coords = torch.rand(Bi, S, N, 2, device="cuda", generator=g) * 70 - 3
    tdim = max(cb.transformer_dim(L, r, 128, False), (2 * 128 + 2 + L * (2 * r + 1) ** 2 + 3) // 4 * 4)
    prev = cb._lib.set_option(cb._lib.OPT_TENSOR_PATH, tensor_path)
    try:
        ctx = torch.autocast("cuda", dtype=torch.bfloat16) if autocast else contextlib.nullcontext()
        with ctx, torch.no_grad():
            blk = cb.CorrBlock(fmaps, num_levels=L, radius=r)
            assert (blk._pyr.split is not None) == tensor_path
            got = cb.TrackTokenizer(blk, coords[:, 0], tdim, num_tracks=counts, num_frames=frames,
                                    frame_index=fi.cuda()).tokens(coords, feats).clone()
            copy = cb.CorrBlock(fmaps.flatten(0, 1)[fi.cuda()], num_levels=L, radius=r)
            want = cb.TrackTokenizer(copy, coords[:, 0], tdim, num_tracks=counts, num_frames=frames).tokens(coords, feats)
            assert torch.equal(got, want)
            plain = cb.TrackTokenizer(blk, coords[:, 0], tdim, frame_index=fi.cuda()).tokens(coords, feats).clone()
            want = cb.TrackTokenizer(copy, coords[:, 0], tdim).tokens(coords, feats)
            assert torch.equal(plain, want)
            for i, (n, s) in enumerate(zip(counts, frames)):
                assert torch.count_nonzero(got[i, n:]) == 0 and torch.count_nonzero(got[i, :, s:]) == 0
    finally:
        cb._lib.set_option(cb._lib.OPT_TENSOR_PATH, prev)
    if tensor_path:
        assert cb._lib.lib.comet_tc_status() == 0


@pytest.mark.gpu
def test_indexed_encoder_matches_gathered_images_and_skips_padded_frames(no_tf32):
    import comet_pose_estimation_b200 as cb

    fnet = load_seeded(cb.ShallowEncoder(input_dim=3).eval(), 3).cuda()
    g = torch.Generator(device="cuda").manual_seed(2)
    S, H, W = 5, 96, 80
    seq_items, fi = _table([5, 2], [[0, 3, 3, 1], [1, 1, 0]], S)    # items (0,0) (0,1) (0,3) (1,0) (1,1)
    counts = [2, 1, 3, 1, 2]
    frames = [5, 5, 5, 2, 2]
    images = torch.randn(2, S, 3, H, W, device="cuda", generator=g)
    images[1, 2:] = float("nan")                                     # padded frames are never read
    tl = (torch.rand(len(counts), S, max(counts), 2, device="cuda", generator=g) * 90 - 10).floor().int()
    seq = torch.tensor([i for i, n in enumerate(counts) for _ in range(n)], device="cuda")
    loc = torch.tensor([j for n in counts for j in range(n)], device="cuda")
    nf = torch.tensor(frames, dtype=torch.int32, device="cuda")
    gathered = images.flatten(0, 1)[fi.cuda()]                        # (items, S, 3, H, W)
    with torch.no_grad():
        got, _ = fnet.encode_packed_patches_of(images, tl[seq, :, loc], seq, num_frames=nf, frame_index=fi.cuda())
        want, _ = fnet.encode_packed_patches_of(gathered, tl[seq, :, loc], seq, num_frames=nf)
    got = got.permute(0, 2, 3, 1).reshape(len(seq), S, 16, 16, 32)
    want = want.permute(0, 2, 3, 1).reshape(len(seq), S, 16, 16, 32)
    live = torch.arange(S, device="cuda")[None, :] < nf[seq][:, None]
    assert torch.equal(got, want)
    assert torch.isfinite(got).all() and torch.count_nonzero(got[~live]) == 0


def _coarse_model():
    import comet_pose_estimation_b200 as cb

    return load_seeded(cb.BaseTrackerPredictor(cfg=cfg(), **cases.FULL_COARSE_CTOR).eval(), cases.FULL_SEEDS["coarse"]).cuda()


def _fine_models():
    import comet_pose_estimation_b200 as cb

    fnet = load_seeded(cb.ShallowEncoder(input_dim=3).eval(), cases.FULL_SEEDS["fnet"]).cuda()
    ftr = load_seeded(cb.BaseTrackerPredictor(cfg=cfg(), **cases.FULL_FINE_CTOR).eval(), cases.FULL_SEEDS["fine"]).cuda()
    return fnet.to(memory_format=torch.channels_last), ftr


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["coarse", "fine"])
@pytest.mark.parametrize("autocast", [False, True])
def test_forward_with_frame_table_equals_gathered_copy(no_tf32, which, autocast):
    g = torch.Generator(device="cuda").manual_seed(3)
    if which == "coarse":
        m, S = _coarse_model(), 16
        _, fi = _table([16, 9], [[0, 5, 15], [0, 8, 3]], S)
        counts, frames = [300, 37, 512, 64, 100, 1], [16, 16, 16, 9, 9, 9]
        fmaps = torch.randn(2, S, 128, 64, 64, device="cuda", generator=g)
        fmaps[1, 9:] = 0.0
        scale, kw = 8.0, dict(down_ratio=2, num_tracks=counts, num_frames=frames)
    else:                            # the fine predictor on ordinary (C = 32, 31 x 31) maps; no counts on this layout
        m, S = _fine_models()[1], 8
        _, fi = _table([8] * 3, [[0, 4], [7], [2, 0, 5]], S)
        counts = [64] * len(fi)
        fmaps = torch.randn(3, S, 32, 31, 31, device="cuda", generator=g)
        scale, kw = 31.0 / 64, {}
    Bi, N = len(counts), max(counts)
    q = torch.rand(Bi, N, 2, device="cuda", generator=g) * 64 * scale
    ctx = torch.autocast("cuda", dtype=torch.bfloat16) if autocast else contextlib.nullcontext()
    with ctx, torch.no_grad():
        got = m(query_points=q, fmaps=fmaps, iters=3, return_feat=True, TRACKorPOSE=False, frame_index=fi.cuda(), **kw)
        want = m(query_points=q, fmaps=fmaps.flatten(0, 1)[fi.cuda()], iters=3, return_feat=True, TRACKorPOSE=False, **kw)
    for i, (a, b) in enumerate(zip(got[0], want[0])):
        assert torch.equal(a, b), i
    for a, b in zip(got[1:], want[1:]):
        assert (a is None and b is None) or torch.equal(a, b)


@pytest.mark.gpu
def test_refine_with_frame_table_equals_gathered_images(no_tf32):
    """The packed patch encoder reads the source images through the table: refine_track is bit-identical to the call on
    the gathered images, score included."""
    import comet_pose_estimation_b200 as cb

    fnet, ftr = _fine_models()
    g = torch.Generator(device="cuda").manual_seed(13)
    S = 8
    _, fi = _table([8, 6], [[0, 3, 7], [5, 0]], S)              # items (0,0) (0,3) (0,7) (1,0) (1,5)
    counts, frames = [40, 7, 64, 1, 30], [8, 8, 8, 6, 6]
    images = torch.rand(2, S, 3, 128, 128, device="cuda", generator=g)
    images[1, 6:] = float("nan")                                  # padded frames are never read
    coarse = torch.rand(len(counts), S, max(counts), 2, device="cuda", generator=g) * 127
    with torch.no_grad():
        got = cb.refine_track(images, fnet, ftr, coarse, compute_score=True, num_tracks=counts, num_frames=frames,
                              frame_index=fi.cuda())
        want = cb.refine_track(images.flatten(0, 1)[fi.cuda()], fnet, ftr, coarse, compute_score=True, num_tracks=counts,
                               num_frames=frames)
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])
    assert torch.isfinite(got[0]).all() and torch.isfinite(got[1]).all()


@pytest.mark.gpu
def test_golden_coarse_case_as_query_frame_zero_item(golden, no_tf32):
    g = golden("tracker_full")
    m = _coarse_model()
    fmaps, q = cases.tracker_case(**cases.FULL_COARSE_CASE)
    fmaps, q = torch.from_numpy(fmaps).cuda(), torch.from_numpy(q).cuda()
    S, N = fmaps.shape[1], q.shape[1]
    H, W = fmaps.shape[-2:]
    scale = cases.FULL_COARSE_CASE["down_ratio"] * 4
    gen = torch.Generator(device="cuda").manual_seed(9)
    src = torch.randn((2,) + tuple(fmaps.shape[1:]), device="cuda", generator=gen)
    src[0] = fmaps[0]
    _, fi = _table([S, S], [[0, 7], [3, 15]], S)            # the golden case is item (0, 0); the others are swapped
    counts = [N, 137, 300, 64]
    qp = torch.rand(4, N, 2, device="cuda", generator=gen) * torch.tensor([W, H], device="cuda") * scale * 0.9
    qp[0] = q[0]
    with torch.no_grad():
        preds, vis, _, _, _ = m(query_points=qp, fmaps=src, iters=cases.FULL_COARSE_ITERS, return_feat=True,
                                down_ratio=cases.FULL_COARSE_CASE["down_ratio"], TRACKorPOSE=False, num_tracks=counts,
                                frame_index=fi.cuda())
    for i in range(cases.FULL_COARSE_ITERS):
        assert rel_to_max(preds[i][0:1].cpu().numpy(), g[f"pred64_{i}"]) <= bar(g[f"pred32_{i}"], g[f"pred64_{i}"]), i
    assert rel_to_max(vis[0:1].cpu().numpy(), g["vis64"]) <= bar(g["vis32"], g["vis64"])
    assert all(torch.isfinite(p).all() for p in preds)


@pytest.mark.gpu
def test_golden_refine_case_as_query_frame_zero_item(golden, no_tf32):
    import comet_pose_estimation_b200 as cb

    r = golden("refine_full")
    fnet, ftr = _fine_models()
    images, _ = cases.refine_case(**cases.FULL_REFINE_CASE)
    images = torch.from_numpy(images).cuda()
    coarse = torch.from_numpy(r["coarse_pred"]).cuda()
    S, N = coarse.shape[1], coarse.shape[2]
    g = torch.Generator(device="cuda").manual_seed(4)
    src = images.repeat(2, 1, 1, 1, 1) + 0.1 * torch.randn((2,) + tuple(images.shape[1:]), device="cuda", generator=g)
    src[0] = images[0]
    _, fi = _table([S, S], [[0, 6], [9]], S)
    counts = [N, 137, 300]
    batch_c = torch.zeros(3, S, N, 2, device="cuda")
    batch_c[0] = coarse[0]
    for i in (1, 2):
        perm = torch.randperm(N, generator=torch.Generator().manual_seed(i))[:counts[i]].cuda()
        batch_c[i, :, :counts[i]] = coarse[0, :, perm] + 3.0
    with torch.no_grad():
        refined, score = cb.refine_track(src, fnet, ftr, batch_c, compute_score=True, num_tracks=counts,
                                         frame_index=fi.cuda())
    inv = cb.inverted_score(score[0:1])
    for k, got in (("refined", refined[0:1]), ("score", score[0:1]), ("inverted", inv)):
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
def test_zero_query_frames_are_bit_identical_to_none(no_tf32):
    tp = _tracker()
    g = torch.Generator(device="cuda").manual_seed(8)
    images = torch.randn(3, 6, 3, 256, 256, device="cuda", generator=g)
    qs = [torch.rand(n, 2, device="cuda", generator=g) * 240 for n in (90, 7, 200)]
    a = tp.track_batch(images, qs, coarse_iters=2)
    b = tp.track_batch(images, qs, coarse_iters=2, query_frames=[torch.zeros(q.shape[0], dtype=torch.int64) for q in qs])
    assert set(b) == set(a) | {"query_frames"} and torch.count_nonzero(b["query_frames"]) == 0
    for k in a:
        _same(a[k], b[k], k)


@pytest.mark.gpu
def test_track_batch_with_query_frames_against_swapped_track_calls(no_tf32):
    """``track_batch(query_frames=...)`` against one ``track()`` per (sequence, query frame) on swapped images.  The two
    arms take their coarse maps from different encoder calls (cuDNN may pick another algorithm for another frame count),
    and the iterated loop amplifies that rounding, so iteration 0 is held within 1e-4 of the maximum, not bitwise; the
    bitwise statements are the kernel, forward and refine tests of this file."""
    import comet_pose_estimation_b200 as cb

    tp = _tracker()
    g = torch.Generator(device="cuda").manual_seed(6)
    frames = [8, 5]
    clips = [torch.randn(s, 3, 512, 512, device="cuda", generator=g) for s in frames]
    qs = [torch.rand(n, 2, device="cuda", generator=g) * 500 for n in (200, 90)]
    qf = [torch.randint(0, s, (q.shape[0],), generator=torch.Generator().manual_seed(s)) for s, q in zip(frames, qs)]
    qf[0][:3] = 0
    out = tp.track_batch(clips, qs, coarse_iters=2, query_frames=qf)
    parts = cb.split_batch(out)
    for b, (p, c, q, t) in enumerate(zip(parts, clips, qs, qf)):
        one = tp.track(c[None], q[None], coarse_iters=2, query_frames=t)
        assert set(p) == set(one)
        for k, v in one.items():
            if isinstance(v, torch.Tensor):
                assert p[k].shape == v.shape, k
        for qq in sorted(set(t.tolist())):
            sel = torch.nonzero(t == qq)[:, 0].cuda()
            ref = tp.track(swap(c[None], qq), q[None, sel], coarse_iters=2)
            want0 = swap(ref["coarse_pred_track_list"][0], qq)
            assert rel_to_max(p["coarse_pred_track_list"][0][:, :, sel].cpu(), want0.cpu()) < 1e-4, (b, qq)
            # the query frame of every track is pinned to its query point
            assert torch.equal(p["coarse_pred_track"][0, qq, sel], q[sel])
        for k, v in out.items():
            if isinstance(v, torch.Tensor) and v.dim() >= 3:
                assert torch.isfinite(v).all(), k


@pytest.mark.gpu
@pytest.mark.parametrize("G", [1, 2, 4])
def test_frames_are_encoded_once(no_tf32, G):
    tp = _tracker()
    seen = []
    h = tp.coarse_fnet.register_forward_hook(lambda mod, inp, out: seen.append(inp[0].shape[0]))
    g = torch.Generator(device="cuda").manual_seed(1)
    frames = [6, 4]
    clips = [torch.randn(s, 3, 256, 256, device="cuda", generator=g) for s in frames]
    qs = [torch.rand(40, 2, device="cuda", generator=g) * 240 for _ in frames]
    qf = [torch.arange(40) % min(G, s) for s in frames]
    try:
        out = tp.track_batch(clips, qs, coarse_iters=1, fine_tracking=False, query_frames=qf)
    finally:
        h.remove()
    assert seen == [sum(frames)]
    assert out["query_frames"][0, :40].tolist() == qf[0].tolist()


@pytest.mark.gpu
def test_graph_replays_for_new_query_frame_sets(no_tf32):
    tp = _tracker()
    g = torch.Generator(device="cuda").manual_seed(7)
    images = torch.randn(2, 6, 3, 256, 256, device="cuda", generator=g)
    qp = torch.rand(2, 100, 2, device="cuda", generator=g) * 240
    first = torch.tensor([[0] * 60 + [2] * 40, [1] * 70 + [5] * 30])
    second = torch.tensor([[4] * 50 + [3] * 50, [0] * 20 + [2] * 80])      # the same (B', N_cap)
    former = tp.coarse_predictor.updateformer
    tp.track_batch(images, qp, coarse_iters=2, fine_tracking=False, query_frames=first)
    captures = getattr(former, "_tc_captures", 0)
    out = tp.track_batch(images, qp, coarse_iters=2, fine_tracking=False, query_frames=second)
    assert getattr(former, "_tc_captures", 0) == captures
    assert torch.isfinite(out["coarse_pred_track"]).all()
