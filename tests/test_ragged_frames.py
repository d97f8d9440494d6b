"""Sequences with different numbers of frames in one call (``track_batch(..., num_frames=...)`` and the ``num_frames``
keyword of every layer below it).  Contract: sequence b of a padded (B, S_max, ...) batch gets what the single-sequence
call on its first S_b frames returns for it alone; every entry of a padded frame or track is exactly 0, and the images
of padded frames are never read.

Kernel-level results are held bitwise to the single-sequence entry points; loop-level results to the float64
reference with the bars of test_full_size.py, plus iteration 0 against the single-sequence run (the iterated loop
amplifies rounding, DESIGN.md section 3)."""
import contextlib
from types import SimpleNamespace as NS

import pytest
import torch

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


# ------------------------------------------------------------------------------------------------ CPU
def _small_former(seed=0):
    from comet_pose_estimation_b200.update_former import EfficientUpdateFormer

    torch.manual_seed(seed)
    return EfficientUpdateFormer(space_depth=2, time_depth=2, input_dim=20, hidden_size=32, num_heads=4, output_dim=6,
                                 num_virtual_tracks=8).eval()


def test_torch_former_with_num_frames_equals_per_sequence_loop():
    m = _small_former()
    x = torch.randn(3, 9, 6, 20)
    counts, frames = [9, 2, 6], [6, 1, 4]
    with torch.no_grad():
        got = m(x, num_tracks=counts, num_frames=frames)
        for b, (n, s) in enumerate(zip(counts, frames)):
            assert torch.equal(got[b:b + 1, :n, :s], m(x[b:b + 1, :n, :s]))
            assert torch.count_nonzero(got[b, n:]) == 0 and torch.count_nonzero(got[b, :, s:]) == 0
        assert torch.equal(m(x, num_tracks=torch.tensor(counts), num_frames=torch.tensor(frames)), got)
        only = m(x, num_frames=frames)
        for b, s in enumerate(frames):
            assert torch.equal(only[b:b + 1, :, :s], m(x[b:b + 1, :, :s]))
            assert torch.count_nonzero(only[b, :, s:]) == 0


@pytest.mark.parametrize("bad", [[0, 3, 3], [3, 7, 3], [3, 3], [3, 3, 3, 3], torch.ones(3, 1, dtype=torch.int64)])
def test_invalid_frame_counts_are_refused(bad):
    import comet_pose_estimation_b200 as cb

    m = _small_former()
    with pytest.raises(AssertionError):
        m(torch.randn(3, 9, 6, 20), num_frames=bad)
    with pytest.raises(AssertionError):
        cb.refine_track(torch.zeros(3, 6, 3, 40, 40), None, None, torch.zeros(3, 6, 9, 2), num_frames=bad)
    with pytest.raises(AssertionError):
        cb.BaseTrackerPredictor(cfg=cfg())(torch.zeros(3, 9, 2), fmaps=torch.zeros(3, 6, 128, 8, 8), TRACKorPOSE=False,
                                           num_frames=bad)


def test_num_frames_needs_track_mode():
    import comet_pose_estimation_b200 as cb

    with pytest.raises(AssertionError):
        cb.BaseTrackerPredictor(cfg=cfg())(torch.zeros(2, 3, 9, 2), fmaps=torch.zeros(2, 3, 128, 8, 8), TRACKorPOSE=True,
                                           num_frames=[3, 2])


def test_split_batch_cuts_both_axes():
    import comet_pose_estimation_b200 as cb

    B, S, N = 3, 5, 7
    counts, frames = [7, 1, 4], [5, 2, 1]
    t = lambda *s: torch.randn(*s)  # noqa: E731
    out = {"coarse_pred_track_list": [t(B, S, N, 2) for _ in range(4)], "coarse_pred_track": t(B, S, N, 2),
           "vis": t(B, S, N), "conf": None, "refine_pred_track": t(B, S, N, 2), "track_score": t(B, S, N),
           "pred_score": t(B, S, N), "num_tracks": torch.tensor(counts), "num_frames": torch.tensor(frames)}
    parts = cb.split_batch(out)
    assert len(parts) == B
    for b, (p, n, s) in enumerate(zip(parts, counts, frames)):
        assert set(p) == set(out) - {"num_tracks", "num_frames"}
        assert p["conf"] is None
        assert len(p["coarse_pred_track_list"]) == 4 and p["coarse_pred_track_list"][2].shape == (1, s, n, 2)
        for k in ("coarse_pred_track", "refine_pred_track"):
            assert p[k].shape == (1, s, n, 2) and torch.equal(p[k][0], out[k][b, :s, :n])
        for k in ("vis", "track_score", "pred_score"):
            assert p[k].shape == (1, s, n)


def test_padded_pred_score_is_normalised_over_real_frames():
    from comet_pose_estimation_b200.refine_track import inverted_score
    from comet_pose_estimation_b200.track_predictor import inverted_score_padded, padded_mask

    counts, frames, S, N = [4, 2], [5, 3], 5, 4
    real = padded_mask(counts, frames, S, N, "cpu")
    score = (torch.rand(2, S, N) + 0.1) * real
    got = inverted_score_padded(score, real)
    assert torch.count_nonzero(got[~real]) == 0
    for b, (n, s) in enumerate(zip(counts, frames)):
        assert torch.equal(got[b:b + 1, :s, :n], inverted_score(score[b:b + 1, :s, :n]))
        assert torch.equal(got[b, :s, :n].max(dim=0)[0], torch.ones(n))
    # the unmasked conversion would make a padded frame's 1 / eps the maximum of the track
    assert inverted_score(score)[1, :3, :2].max() < 1e-3


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture
def no_tf32():
    a, b = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = a, b


LENGTHS = (1, 2, 15, 16, 17, 32, 33, 63, 64, 72)
# problem counts of the single call: at np = 3, 72 frames and 8 heads the key-split kernel serves up to 37 problems
GROUPS = (8, 40)


@pytest.mark.gpu
@pytest.mark.parametrize("np_", [1, 3])
@pytest.mark.parametrize("D", [384, 256])          # dh = 48 (coarse), 32 (fine)
def test_varlen_time_attention_bit_identical_per_track(np_, D):
    """One varlen call over tracks of every (length, group) pair vs one comet_attention_planes_f32 call per pair."""
    from comet_pose_estimation_b200 import update_former_tc as tc

    H, T = 8, max(LENGTHS)
    dh, ld, od = D // H, 3 * D, tc._ceil8(D)
    run = tc._Run(tc._Weights(), np_, torch.device("cuda"))
    seqs = [(L, g) for L in LENGTHS for g in GROUPS]
    ntr = sum(g for _, g in seqs)
    gen = torch.Generator(device="cuda").manual_seed(11)
    qkv = torch.randn(ntr * T, ld, device="cuda", generator=gen)
    lens = torch.tensor([L for L, g in seqs for _ in range(g)], dtype=torch.int32, device="cuda")
    grp = torch.tensor([g for _, g in seqs for _ in range(g)], dtype=torch.int32, device="cuda")
    off = torch.arange(ntr, dtype=torch.int32, device="cuda") * T
    got = run.attention_varlen(qkv[:, :D], qkv[:, D:2 * D], qkv[:, 2 * D:], H, dh, 1, ntr, off, lens, off, lens, (1, T),
                               (1, T), (grp, min(GROUPS), max(GROUPS)), ntr * T, D, zero=True)
    t0 = 0
    for L, g in seqs:
        rows = slice(t0 * T, (t0 + g) * T)
        q = qkv[rows]
        want = run.attention(q[:, :D], q[:, D:2 * D], q[:, 2 * D:], g, H, L, L, dh, T * ld, ld, T * ld, ld, g * T, D,
                             T * od, od)
        mine = got[:, rows].reshape(got.shape[0], g, T, -1)
        assert torch.equal(mine[:, :, :L], want.reshape(want.shape[0], g, T, -1)[:, :, :L]), (L, g)
        assert torch.count_nonzero(mine[:, :, L:]) == 0
        t0 += g


@pytest.mark.gpu
@pytest.mark.parametrize("tensor_path", [True, False])
@pytest.mark.parametrize("autocast", [False, True])
def test_coarse_tokens_with_frame_and_track_counts(no_tf32, tensor_path, autocast):
    """Tensor and SIMT paths: rows of real (track, frame) pairs bit-identical to the single-sequence call on its first S_b
    frames, padded rows exactly 0, and NaN in the features of padded frames is never read."""
    import comet_pose_estimation_b200 as cb

    if tensor_path and not cb._lib.lib.comet_has_tensor_path():
        pytest.skip("no sm_100 tensor path on this device")
    g = torch.Generator(device="cuda").manual_seed(5)
    counts, frames, S, L, r = [300, 137, 1, 64], [5, 2, 5, 1], 5, 4, 3
    B, N = len(counts), max(counts)
    fmaps = torch.randn(B, S, 128, 64, 64, device="cuda", generator=g)
    feats = torch.randn(B, S, N, 128, device="cuda", generator=g)
    coords = torch.rand(B, S, N, 2, device="cuda", generator=g) * 70 - 3
    feats_nan = feats.clone()
    for b, s in enumerate(frames):
        feats_nan[b, s:] = float("nan")
        coords[b, s:] = 0.0
    tdim = max(cb.transformer_dim(L, r, 128, False), (2 * 128 + 2 + L * (2 * r + 1) ** 2 + 3) // 4 * 4)
    prev = cb._lib.set_option(cb._lib.OPT_TENSOR_PATH, tensor_path)
    try:
        ctx = torch.autocast("cuda", dtype=torch.bfloat16) if autocast else contextlib.nullcontext()
        with ctx, torch.no_grad():
            blk = cb.CorrBlock(fmaps, num_levels=L, radius=r)
            assert (blk._pyr.split is not None) == tensor_path
            tok = cb.TrackTokenizer(blk, coords[:, 0], tdim, num_tracks=counts, num_frames=frames)
            got = tok.tokens(coords, feats_nan).clone()
            only = cb.TrackTokenizer(blk, coords[:, 0], tdim, num_frames=frames).tokens(coords, feats_nan).clone()
            for b, (n, s) in enumerate(zip(counts, frames)):
                one = cb.CorrBlock(fmaps[b:b + 1, :s], num_levels=L, radius=r)
                want = cb.TrackTokenizer(one, coords[b:b + 1, 0, :n], tdim).tokens(coords[b:b + 1, :s, :n],
                                                                                    feats[b:b + 1, :s, :n])
                assert torch.equal(got[b:b + 1, :n, :s], want), (b, n, s)
                assert torch.count_nonzero(got[b, n:]) == 0 and torch.count_nonzero(got[b, :, s:]) == 0
                assert torch.equal(only[b:b + 1, :n, :s], want) and torch.count_nonzero(only[b, :, s:]) == 0
    finally:
        cb._lib.set_option(cb._lib.OPT_TENSOR_PATH, prev)
    if tensor_path:
        assert cb._lib.lib.comet_tc_status() == 0


@pytest.mark.gpu
@pytest.mark.parametrize("autocast", [False, True])
def test_fine_up2_tokens_with_frame_counts(no_tf32, autocast):
    """The fine tracker's lookup on the encoder's half-resolution map (COMET_PYR_UP2_SOURCE): one packed track per
    sequence, each with its own frame count."""
    import comet_pose_estimation_b200 as cb

    g = torch.Generator(device="cuda").manual_seed(12)
    frames, S, L, r = [6, 1, 3, 6, 2], 6, 3, 3
    P = len(frames)
    src = torch.randn(P, S, 16, 16, 32, device="cuda", generator=g).permute(0, 1, 4, 2, 3)   # channels-last maps
    feats = torch.randn(P, S, 1, 32, device="cuda", generator=g)
    coords = torch.rand(P, S, 1, 2, device="cuda", generator=g) * 34 - 2
    tdim = cb.transformer_dim(L, r, 32, fine=True)
    ctx = torch.autocast("cuda", dtype=torch.bfloat16) if autocast else contextlib.nullcontext()
    with ctx, torch.no_grad():
        up = cb.Upsampled2x(src)
        blk = cb.CorrBlock(up, num_levels=L, radius=r)
        got = cb.TrackTokenizer(blk, coords[:, 0], tdim, num_frames=frames).tokens(coords, feats).clone()
        for p, s in enumerate(frames):
            one = cb.CorrBlock(cb.Upsampled2x(src[p:p + 1, :s]), num_levels=L, radius=r)
            want = cb.TrackTokenizer(one, coords[p:p + 1, 0], tdim).tokens(coords[p:p + 1, :s], feats[p:p + 1, :s])
            assert torch.equal(got[p:p + 1, :, :s], want), (p, s)
            assert torch.count_nonzero(got[p, :, s:]) == 0


@pytest.mark.gpu
def test_varlen_encoder_matches_ragged_and_skips_padded_frames(no_tf32):
    import comet_pose_estimation_b200 as cb

    fnet = load_seeded(cb.ShallowEncoder(input_dim=3).eval(), 3).cuda()
    g = torch.Generator(device="cuda").manual_seed(2)
    B, S, H, W = 3, 5, 96, 80
    counts, frames = [5, 1, 3], [5, 2, 3]
    images = torch.randn(B, S, 3, H, W, device="cuda", generator=g)
    tl = (torch.rand(B, S, max(counts), 2, device="cuda", generator=g) * 90 - 10).floor().int()
    seq = torch.tensor([b for b, n in enumerate(counts) for _ in range(n)], device="cuda")
    loc = torch.tensor([j for n in counts for j in range(n)], device="cuda")
    nf = torch.tensor(frames, dtype=torch.int32, device="cuda")
    poisoned = images.clone()
    for b, s in enumerate(frames):
        poisoned[b, s:] = float("nan")
    with torch.no_grad():
        want, _ = fnet.encode_packed_patches_of(images, tl[seq, :, loc], seq)
        got, _ = fnet.encode_packed_patches_of(poisoned, tl[seq, :, loc], seq, num_frames=nf)
    want = want.permute(0, 2, 3, 1).reshape(len(seq), S, 16, 16, 32)
    got = got.permute(0, 2, 3, 1).reshape(len(seq), S, 16, 16, 32)
    live = torch.arange(S, device="cuda")[None, :] < nf[seq][:, None]
    assert torch.equal(got[live], want[live])
    assert torch.count_nonzero(got[~live]) == 0


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
def test_ragged_frames_transformer_matches_single_sequence(no_tf32, which, autocast):
    m = (_coarse_model() if which == "coarse" else _fine_models()[1]).updateformer
    g = torch.Generator(device="cuda").manual_seed(3)
    if which == "coarse":
        counts, frames = [300, 37, 512, 64], [16, 9, 12, 1]
        counts2, frames2 = [12, 500, 290, 100], [3, 16, 7, 16]
    else:                           # the fine tracker: packed tracks, one track per sequence
        counts, frames = None, [16, 9, 12, 1, 16, 5, 2, 14]
        counts2, frames2 = None, [4, 16, 16, 8, 3, 11, 16, 1]
    B = len(frames)
    N = 1 if counts is None else max(counts)
    x = torch.randn(B, N, 16, m.input_transform.in_features, device="cuda", generator=g)
    ctx = torch.autocast("cuda", dtype=torch.bfloat16) if autocast else contextlib.nullcontext()
    with ctx, torch.no_grad():
        got = m(x, num_tracks=counts, num_frames=frames)
        captures = getattr(m, "_tc_captures", 0)
        got2 = m(x, num_tracks=counts2, num_frames=frames2)          # new counts replay the captured graph
        assert getattr(m, "_tc_captures", 0) == captures
        for out, cs, fs in ((got, counts, frames), (got2, counts2, frames2)):
            for b, s in enumerate(fs):
                n = N if cs is None else cs[b]
                want = m(x[b:b + 1, :n, :s])
                # every item runs the kernel family and arithmetic of its single call, and row-wise kernels do not
                # depend on the row count, so the rows are bit-identical
                assert torch.equal(out[b:b + 1, :n, :s], want), (b, n, s)
                assert torch.count_nonzero(out[b, n:]) == 0 and torch.count_nonzero(out[b, :, s:]) == 0


@pytest.mark.gpu
def test_golden_coarse_case_inside_ragged_frames_batch(golden, no_tf32):
    g = golden("tracker_full")
    m = _coarse_model()
    fmaps, q = cases.tracker_case(**cases.FULL_COARSE_CASE)
    fmaps, q = torch.from_numpy(fmaps).cuda(), torch.from_numpy(q).cuda()
    S, N = fmaps.shape[1], q.shape[1]
    H, W = fmaps.shape[-2:]
    scale = cases.FULL_COARSE_CASE["down_ratio"] * 4
    gen = torch.Generator(device="cuda").manual_seed(9)
    frames, counts = [9, S, 12], [137, N, 300]
    qp = torch.zeros(3, N, 2, device="cuda")
    fm = torch.randn((3,) + tuple(fmaps.shape[1:]), device="cuda", generator=gen)
    fm[1] = fmaps[0]
    for b in (0, 2):
        qp[b, :counts[b]] = torch.rand(counts[b], 2, device="cuda", generator=gen) * torch.tensor([W, H], device="cuda") * scale * 0.9
        fm[b, frames[b]:] = 0.0            # what track_batch's encoder leaves in padded frames
    qp[1] = q[0]
    kw = dict(iters=cases.FULL_COARSE_ITERS, return_feat=True, down_ratio=cases.FULL_COARSE_CASE["down_ratio"],
              TRACKorPOSE=False)
    with torch.no_grad():
        preds, vis, feats, qfeat, _ = m(query_points=qp, fmaps=fm, num_tracks=counts, num_frames=frames, **kw)
        for i in range(cases.FULL_COARSE_ITERS):
            r32, r64 = g[f"pred32_{i}"], g[f"pred64_{i}"]
            assert rel_to_max(preds[i][1:2].cpu().numpy(), r64) <= bar(r32, r64), i
        assert rel_to_max(vis[1:2].cpu().numpy(), g["vis64"]) <= bar(g["vis32"], g["vis64"])
        for b in (0, 2):
            n, s = counts[b], frames[b]
            one = m(query_points=qp[b:b + 1, :n], fmaps=fm[b:b + 1, :s], **kw)
            assert rel_to_max(preds[0][b:b + 1, :s, :n].cpu(), one[0][0].cpu()) < 1e-4, b
            for p in preds:
                assert torch.isfinite(p).all()
                assert torch.count_nonzero(p[b, s:]) == 0 and torch.count_nonzero(p[b, :, n:]) == 0
            assert torch.count_nonzero(vis[b, s:]) == 0


@pytest.mark.gpu
def test_golden_refine_case_inside_ragged_frames_batch(golden, no_tf32):
    import comet_pose_estimation_b200 as cb

    r = golden("refine_full")
    fnet, ftr = _fine_models()
    images, _ = cases.refine_case(**cases.FULL_REFINE_CASE)
    images = torch.from_numpy(images).cuda()
    coarse = torch.from_numpy(r["coarse_pred"]).cuda()
    S, N = coarse.shape[1], coarse.shape[2]
    g = torch.Generator(device="cuda").manual_seed(4)
    frames, counts = [9, S, 12], [137, N, 300]
    batch_c = torch.zeros(3, S, N, 2, device="cuda")
    batch_c[1] = coarse[0]
    batch_i = images.repeat(3, 1, 1, 1, 1) + 0.1 * torch.randn((3,) + tuple(images.shape[1:]), device="cuda", generator=g)
    batch_i[1] = images[0]
    for b in (0, 2):
        perm = torch.randperm(N, generator=torch.Generator().manual_seed(b))[:counts[b]].cuda()
        batch_c[b, :frames[b], :counts[b]] = coarse[0, :frames[b], perm] + 3.0
        batch_i[b, frames[b]:] = float("nan")                   # padded frames are never read
    with torch.no_grad():
        refined, score = cb.refine_track(batch_i, fnet, ftr, batch_c, compute_score=True, num_tracks=counts,
                                         num_frames=frames)
        inv = cb.inverted_score(score[1:2])
        for k, got in (("refined", refined[1:2]), ("score", score[1:2]), ("inverted", inv)):
            assert rel_to_max(got.cpu().numpy(), r[k + "64"]) <= bar(r[k + "32"], r[k + "64"]), k
        assert torch.isfinite(refined).all() and torch.isfinite(score).all()
        for b in (0, 2):
            n, s = counts[b], frames[b]
            assert torch.count_nonzero(refined[b, s:]) == 0 and torch.count_nonzero(score[b, s:]) == 0
            assert torch.count_nonzero(refined[b, :, n:]) == 0 and torch.count_nonzero(score[b, :, n:]) == 0
            one_r, one_s = cb.refine_track(batch_i[b:b + 1, :s], fnet, ftr, batch_c[b:b + 1, :s, :n], compute_score=True)
            assert rel_to_max(refined[b:b + 1, :s, :n].cpu(), one_r.cpu()) < 1e-3, b
            assert rel_to_max(score[b:b + 1, :s, :n].cpu(), one_s.cpu()) < 1e-3, b


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
def test_full_frame_counts_are_bit_identical_to_no_frame_counts(no_tf32):
    tp = _tracker()
    g = torch.Generator(device="cuda").manual_seed(8)
    images = torch.randn(3, 6, 3, 256, 256, device="cuda", generator=g)
    qs = [torch.rand(n, 2, device="cuda", generator=g) * 240 for n in (90, 7, 200)]
    a = tp.track_batch(images, qs, coarse_iters=2)
    b = tp.track_batch(images, qs, coarse_iters=2, num_frames=[6, 6, 6])
    assert set(b) == set(a) | {"num_frames"}
    for k in a:
        _same(a[k], b[k], k)


@pytest.mark.gpu
def test_track_batch_ragged_frames_from_images(no_tf32):
    import comet_pose_estimation_b200 as cb

    tp = _tracker()
    g = torch.Generator(device="cuda").manual_seed(6)
    frames = [6, 3, 5]
    clips = [torch.randn(s, 3, 256, 256, device="cuda", generator=g) for s in frames]
    qs = [torch.rand(n, 2, device="cuda", generator=g) * 240 for n in (90, 7, 200)]
    out = tp.track_batch(clips, qs, coarse_iters=2)
    assert out["num_frames"].tolist() == frames
    padded = torch.full((3, 6, 3, 256, 256), float("nan"), device="cuda")
    for b, c in enumerate(clips):
        padded[b, :c.shape[0]] = c
    out2 = tp.track_batch(padded, qs, coarse_iters=2, num_frames=frames)   # NaN in every padded frame
    for k in out:
        _same(out[k], out2[k], k)
    parts = cb.split_batch(out)
    for b, (p, q, c) in enumerate(zip(parts, qs, clips)):
        n, s = q.shape[0], c.shape[0]
        one = tp.track(c[None], q[None], coarse_iters=2)
        assert set(p) == set(one)
        for k, v in one.items():
            if isinstance(v, torch.Tensor):
                assert p[k].shape == v.shape, k
        # the encoder's cuDNN algorithm may differ with the batch size, so later iterations are not held bitwise
        assert rel_to_max(p["coarse_pred_track_list"][0].cpu(), one["coarse_pred_track_list"][0].cpu()) < 1e-4, b
        for k, v in out.items():
            if isinstance(v, torch.Tensor) and v.dim() >= 3:
                assert torch.isfinite(v).all(), k
                assert torch.count_nonzero(v[b, s:]) == 0 and torch.count_nonzero(v[b, :, n:]) == 0, k
        assert torch.equal(p["pred_score"][0].max(dim=0)[0], torch.ones(n, device="cuda"))
