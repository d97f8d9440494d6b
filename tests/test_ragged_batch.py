"""Ragged batching: several sequences with different track counts in one call (``TrackerPredictor.track_batch`` and the
``num_tracks`` keyword of every layer below it).  Contract: sequence b of a batch gets what the single-sequence call
returns for it alone; every padded entry (track n >= N_b) is exactly 0.

Kernel-level results are held bitwise to the single-sequence entry points.  The iterated tracker loop amplifies
rounding ~200x per iteration (DESIGN.md section 3), so loop-level results are held to the float64 reference with the
bars of test_full_size.py, plus iteration 0 against the single-sequence run."""
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


def test_torch_former_with_num_tracks_equals_per_sequence_loop():
    m = _small_former()
    x = torch.randn(3, 9, 5, 20)
    counts = [9, 2, 6]
    with torch.no_grad():
        got = m(x, num_tracks=counts)
        for b, n in enumerate(counts):
            want = m(x[b:b + 1, :n])
            assert torch.equal(got[b:b + 1, :n], want)
            assert torch.count_nonzero(got[b, n:]) == 0
        assert torch.equal(m(x, num_tracks=torch.tensor(counts)), got)


@pytest.mark.parametrize("bad", [[0, 3, 3], [3, 10, 3], [3, 3], [3, 3, 3, 3], torch.ones(3, 1, dtype=torch.int64)])
def test_invalid_counts_are_refused(bad):
    import comet_pose_estimation_b200 as cb

    m = _small_former()
    with pytest.raises(AssertionError):
        m(torch.randn(3, 9, 5, 20), num_tracks=bad)
    with pytest.raises(AssertionError):
        cb.refine_track(torch.zeros(3, 2, 3, 40, 40), None, None, torch.zeros(3, 2, 9, 2), num_tracks=bad)
    with pytest.raises(AssertionError):
        cb.BaseTrackerPredictor(cfg=cfg())(torch.zeros(3, 9, 2), fmaps=torch.zeros(3, 2, 128, 8, 8), TRACKorPOSE=False,
                                           num_tracks=bad)


def test_num_tracks_needs_track_mode():
    import comet_pose_estimation_b200 as cb

    with pytest.raises(AssertionError):
        cb.BaseTrackerPredictor(cfg=cfg())(torch.zeros(2, 3, 9, 2), fmaps=torch.zeros(2, 3, 128, 8, 8), TRACKorPOSE=True,
                                           num_tracks=[9, 4])


def test_split_batch_keys_and_shapes():
    import comet_pose_estimation_b200 as cb

    B, S, N = 3, 4, 7
    counts = [7, 1, 4]
    t = lambda *s: torch.randn(*s)  # noqa: E731
    out = {"coarse_pred_track_list": [t(B, S, N, 2) for _ in range(4)], "coarse_pred_track": t(B, S, N, 2),
           "vis": t(B, S, N), "conf": None, "refine_pred_track": t(B, S, N, 2), "track_score": t(B, S, N),
           "pred_score": t(B, S, N), "num_tracks": torch.tensor(counts)}
    parts = cb.split_batch(out)
    assert len(parts) == B
    for b, (p, n) in enumerate(zip(parts, counts)):
        assert set(p) == set(out) - {"num_tracks"}
        assert p["conf"] is None
        assert len(p["coarse_pred_track_list"]) == 4 and p["coarse_pred_track_list"][2].shape == (1, S, n, 2)
        for k in ("coarse_pred_track", "refine_pred_track"):
            assert p[k].shape == (1, S, n, 2) and torch.equal(p[k][0], out[k][b, :, :n])
        for k in ("vis", "track_score", "pred_score"):
            assert p[k].shape == (1, S, n)


@pytest.mark.parametrize("world", [1, 2, 3])
@pytest.mark.parametrize("batch_size", [1, 2, 4])
def test_run_sharded_batched_covers_every_index_once(world, batch_size):
    from comet_pose_estimation_b200.launch import run_sharded, run_sharded_batched

    items = [f"seq{i}" for i in range(11)]
    seen = {}
    for rank in range(world):
        calls = []

        def fn(batch):
            calls.append(len(batch))
            return [s.upper() for s in batch]

        got = run_sharded_batched(items, fn, batch_size, rank=rank, world=world)
        assert max(calls) <= batch_size
        assert got == run_sharded(items, str.upper, rank=rank, world=world)
        assert not seen.keys() & got.keys()
        seen.update(got)
    assert sorted(seen) == list(range(len(items)))
    assert all(seen[i] == items[i].upper() for i in seen)


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture
def no_tf32():
    a, b = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = a, b


COUNTS = (512, 137, 300, 1)


def _ragged_token_inputs(g, S=3, L=4, r=3):
    B, N = len(COUNTS), max(COUNTS)
    fmaps = torch.randn(B, S, 128, 64, 64, device="cuda", generator=g)
    feats = torch.randn(B, S, N, 128, device="cuda", generator=g)
    coords = torch.rand(B, S, N, 2, device="cuda", generator=g) * 70 - 3
    return fmaps, feats, coords, L, r


@pytest.mark.gpu
@pytest.mark.parametrize("tensor_path", [True, False])
@pytest.mark.parametrize("autocast", [False, True])
def test_ragged_tokens_bit_identical_per_sequence(no_tf32, tensor_path, autocast):
    import comet_pose_estimation_b200 as cb

    if tensor_path and not cb._lib.lib.comet_has_tensor_path():
        pytest.skip("no sm_100 tensor path on this device")
    g = torch.Generator(device="cuda").manual_seed(5)
    fmaps, feats, coords, L, r = _ragged_token_inputs(g)
    tdim = max(cb.transformer_dim(L, r, 128, False), (2 * 128 + 2 + L * (2 * r + 1) ** 2 + 3) // 4 * 4)
    prev = cb._lib.set_option(cb._lib.OPT_TENSOR_PATH, tensor_path)
    try:
        ctx = torch.autocast("cuda", dtype=torch.bfloat16) if autocast else contextlib.nullcontext()
        with ctx, torch.no_grad():
            blk = cb.CorrBlock(fmaps, num_levels=L, radius=r)
            assert (blk._pyr.split is not None) == tensor_path
            tok = cb.TrackTokenizer(blk, coords[:, 0], tdim, num_tracks=list(COUNTS)).tokens(coords, feats).clone()
            for b, n in enumerate(COUNTS):
                one = cb.CorrBlock(fmaps[b:b + 1], num_levels=L, radius=r)
                want = cb.TrackTokenizer(one, coords[b:b + 1, 0, :n], tdim).tokens(coords[b:b + 1, :, :n],
                                                                                    feats[b:b + 1, :, :n])
                assert torch.equal(tok[b:b + 1, :n], want), (b, n)
                assert torch.count_nonzero(tok[b, n:]) == 0
    finally:
        cb._lib.set_option(cb._lib.OPT_TENSOR_PATH, prev)
    if tensor_path:
        assert cb._lib.lib.comet_tc_status() == 0


@pytest.mark.gpu
def test_ragged_encoder_maps_bit_identical(no_tf32):
    import comet_pose_estimation_b200 as cb

    fnet = load_seeded(cb.ShallowEncoder(input_dim=3).eval(), 3).cuda()
    g = torch.Generator(device="cuda").manual_seed(2)
    B, S, H, W = 3, 4, 96, 80
    counts = [5, 1, 3]
    images = torch.randn(B, S, 3, H, W, device="cuda", generator=g)
    tl = (torch.rand(B, S, max(counts), 2, device="cuda", generator=g) * 90 - 10).floor().int()
    seq = torch.tensor([b for b, n in enumerate(counts) for _ in range(n)], device="cuda")
    loc = torch.tensor([j for n in counts for j in range(n)], device="cuda")
    with torch.no_grad():
        got, _ = fnet.encode_packed_patches_of(images, tl[seq, :, loc], seq)            # (P*S, C, 16, 16)
        got = got.permute(0, 2, 3, 1).reshape(len(seq), S, 16, 16, 32)
        for b, n in enumerate(counts):
            want, _ = fnet.encode_patches_of(images[b:b + 1], tl[b:b + 1, :, :n])      # (n*S, C, 16, 16), (n, s) order
            want = want.permute(0, 2, 3, 1).reshape(n, S, 16, 16, 32)
            assert torch.equal(got[seq == b], want), b


def _attention_case(g, np_, counts, T=4, V=64, D=384, H=8):
    """Per-sequence single calls of comet_attention_planes_f32 vs one varlen call, all three space-attention shapes."""
    from comet_pose_estimation_b200 import update_former_tc as tc

    run = tc._Run(tc._Weights(), np_, torch.device("cuda"))
    B, Nc = len(counts), (max(counts) + 63) // 64 * 64
    pts = torch.randn(B * Nc * T, 3 * D, device="cuda", generator=g)
    vir = torch.randn(B * V * T, 3 * D, device="cuda", generator=g)
    lay = tc._RaggedLayout(torch.tensor(counts, dtype=torch.int32, device="cuda"), B, Nc, V, T)
    dh, ld = D // H, 3 * D
    cases_ = []
    # virtual -> points, points -> virtual, virtual self attention
    got = run.attention_varlen(vir[:, :D], pts[:, D:2 * D], pts[:, 2 * D:], H, dh, T, lay.items, lay.vir_off, lay.vir_len,
                               lay.pts_off, lay.pts_len, (V, V), (1, Nc), T, B * V * T, D)
    cases_.append(("v2p", got, vir, pts, lambda b: (V, counts[b])))
    got = run.attention_varlen(pts[:, :D], vir[:, D:2 * D], vir[:, 2 * D:], H, dh, T, lay.items, lay.pts_off, lay.pts_len,
                               lay.vir_off, lay.vir_len, (1, Nc), (V, V), T, B * Nc * T, D, zero=True)
    cases_.append(("p2v", got, pts, vir, lambda b: (counts[b], V)))
    got = run.attention_varlen(vir[:, :D], vir[:, D:2 * D], vir[:, 2 * D:], H, dh, T, lay.items, lay.vir_off, lay.vir_len,
                               lay.vir_off, lay.vir_len, (V, V), (V, V), T, B * V * T, D)
    cases_.append(("vv", got, vir, vir, lambda b: (V, V)))
    for name, got, qsrc, ksrc, lens in cases_:
        qn = qsrc.shape[0] // (B * T)
        kn = ksrc.shape[0] // (B * T)
        for b in range(B):
            Lq, Lk = lens(b)
            q = qsrc[b * qn * T:(b * qn + Lq) * T]
            k = ksrc[b * kn * T:(b * kn + Lk) * T]
            want = run.attention(q[:, :D], k[:, D:2 * D], k[:, 2 * D:], T, H, Lq, Lk, dh, ld, T * ld, ld, T * ld, Lq * T, D,
                                 tc._ceil8(D), T * tc._ceil8(D))
            rows = got[:, b * qn * T:(b * qn + Lq) * T]
            assert torch.equal(rows, want), (name, b, Lq, Lk)
            if name == "p2v":
                assert torch.count_nonzero(got[:, (b * qn + Lq) * T:(b + 1) * qn * T]) == 0


@pytest.mark.gpu
@pytest.mark.parametrize("np_", [1, 3])
def test_varlen_attention_bit_identical_per_item(np_):
    g = torch.Generator(device="cuda").manual_seed(7)
    _attention_case(g, np_, [200, 17, 64, 65, 1, 130])


def _coarse_model():
    import comet_pose_estimation_b200 as cb

    return load_seeded(cb.BaseTrackerPredictor(cfg=cfg(), **cases.FULL_COARSE_CTOR).eval(), cases.FULL_SEEDS["coarse"]).cuda()


@pytest.mark.gpu
@pytest.mark.parametrize("autocast", [False, True])
def test_ragged_transformer_forward_matches_single_sequence(no_tf32, autocast):
    m = _coarse_model().updateformer
    g = torch.Generator(device="cuda").manual_seed(3)
    counts = [300, 37, 512, 64]
    x = torch.randn(len(counts), max(counts), 16, m.input_transform.in_features, device="cuda", generator=g)
    ctx = torch.autocast("cuda", dtype=torch.bfloat16) if autocast else contextlib.nullcontext()
    tol = 2e-3 if autocast else 1e-6
    exact = []
    with ctx, torch.no_grad():
        got = m(x, num_tracks=counts)
        # another batch with other counts replays the same captured graph
        captures = getattr(m, "_tc_captures", 0)
        counts2 = [12, 500, 290, 100]
        got2 = m(x, num_tracks=counts2)
        assert getattr(m, "_tc_captures", 0) == captures
        for b, n in enumerate(counts):
            want = m(x[b:b + 1, :n])
            assert rel_to_max(got[b:b + 1, :n].cpu(), want.cpu()) <= tol, b
            exact.append(bool(torch.equal(got[b:b + 1, :n], want)))
            assert torch.count_nonzero(got[b, n:]) == 0
        want2 = m(x[1:2, :500])
        assert rel_to_max(got2[1:2, :500].cpu(), want2.cpu()) <= tol
    print(f"ragged transformer bit-identical per sequence (autocast={autocast}): {exact}")


def _golden_tracker_batch(golden, slot_n=(137, 300)):
    """Batch of three: slot 1 is the golden full-size coarse case, slots 0 / 2 seeded sequences of N = 137 / 300."""
    fmaps, q = cases.tracker_case(**cases.FULL_COARSE_CASE)
    fmaps, q = torch.from_numpy(fmaps).cuda(), torch.from_numpy(q).cuda()
    g = torch.Generator(device="cuda").manual_seed(9)
    N = q.shape[1]
    H, W = fmaps.shape[-2:]
    scale = cases.FULL_COARSE_CASE["down_ratio"] * 4
    qs, fs = [], []
    for n in slot_n:
        qs.append(torch.rand(1, n, 2, device="cuda", generator=g) * torch.tensor([W, H], device="cuda") * scale * 0.9)
        fs.append(torch.randn(fmaps.shape, device="cuda", generator=g))
    counts = [slot_n[0], N, slot_n[1]]
    qp = torch.zeros(3, max(counts), 2, device="cuda")
    qp[0, :counts[0]], qp[1, :N], qp[2, :counts[2]] = qs[0][0], q[0], qs[1][0]
    return torch.cat([fs[0], fmaps, fs[1]]), qp, counts, (fs, qs)


@pytest.mark.gpu
def test_golden_coarse_case_inside_ragged_batch(golden, no_tf32):
    g, gf = golden("tracker_full"), golden("tracker_full_feats")
    m = _coarse_model()
    fmaps, qp, counts, (fs, qs) = _golden_tracker_batch(golden)
    kw = dict(iters=cases.FULL_COARSE_ITERS, return_feat=True, down_ratio=cases.FULL_COARSE_CASE["down_ratio"],
              TRACKorPOSE=False)
    with torch.no_grad():
        preds, vis, feats, qfeat, _ = m(query_points=qp, fmaps=fmaps, num_tracks=counts, **kw)
        N = counts[1]
        for i in range(cases.FULL_COARSE_ITERS):
            r32, r64 = g[f"pred32_{i}"], g[f"pred64_{i}"]
            assert rel_to_max(preds[i][1:2, :, :N].cpu().numpy(), r64) <= bar(r32, r64), i
        assert rel_to_max(qfeat[1:2, :N].cpu().numpy(), gf["query_feat32"]) < 1e-5
        assert rel_to_max(vis[1:2, :, :N].cpu().numpy(), g["vis64"]) <= bar(g["vis32"], g["vis64"])
        for slot, (f, q) in zip((0, 2), zip(fs, qs)):
            n = counts[slot]
            one = m(query_points=q, fmaps=f, **kw)
            assert rel_to_max(preds[0][slot:slot + 1, :, :n].cpu(), one[0][0].cpu()) < 1e-5, slot
            for p in preds:
                assert torch.isfinite(p).all()
                assert torch.count_nonzero(p[slot, :, n:]) == 0
        assert torch.isfinite(vis).all() and torch.count_nonzero(vis[0, :, counts[0]:]) == 0


def _fine_models():
    import comet_pose_estimation_b200 as cb

    fnet = load_seeded(cb.ShallowEncoder(input_dim=3).eval(), cases.FULL_SEEDS["fnet"]).cuda()
    ftr = load_seeded(cb.BaseTrackerPredictor(cfg=cfg(), **cases.FULL_FINE_CTOR).eval(), cases.FULL_SEEDS["fine"]).cuda()
    return fnet.to(memory_format=torch.channels_last), ftr


@pytest.mark.gpu
def test_golden_refine_case_inside_ragged_batch(golden, no_tf32):
    import comet_pose_estimation_b200 as cb

    r = golden("refine_full")
    fnet, ftr = _fine_models()
    images, _ = cases.refine_case(**cases.FULL_REFINE_CASE)
    images = torch.from_numpy(images).cuda()
    coarse = torch.from_numpy(r["coarse_pred"]).cuda()
    N = coarse.shape[2]
    g = torch.Generator(device="cuda").manual_seed(4)
    other = coarse[:, :, torch.randperm(N, generator=torch.Generator().manual_seed(1))[:137].cuda()] + 3.0
    counts = [137, N]
    batch_c = torch.zeros(2, coarse.shape[1], N, 2, device="cuda")
    batch_c[0, :, :137], batch_c[1] = other[0], coarse[0]
    batch_i = torch.cat([images + 0.1 * torch.randn(images.shape, device="cuda", generator=g), images])
    with torch.no_grad():
        refined, score = cb.refine_track(batch_i, fnet, ftr, batch_c, compute_score=True, num_tracks=counts)
        inv = cb.inverted_score(score[1:2])
        for k, got in (("refined", refined[1:2]), ("score", score[1:2]), ("inverted", inv)):
            assert rel_to_max(got.cpu().numpy(), r[k + "64"]) <= bar(r[k + "32"], r[k + "64"]), k
    assert torch.isfinite(refined).all() and torch.isfinite(score).all()
    assert torch.count_nonzero(refined[0, :, 137:]) == 0 and torch.count_nonzero(score[0, :, 137:]) == 0


def _tracker():
    import comet_pose_estimation_b200 as cb

    torch.manual_seed(0)
    return cb.TrackerPredictor().eval().cuda()


@pytest.mark.gpu
def test_single_sequence_batch_is_bit_identical_to_track(no_tf32):
    import comet_pose_estimation_b200 as cb

    tp = _tracker()
    g = torch.Generator(device="cuda").manual_seed(8)
    images = torch.randn(1, 4, 3, 256, 256, device="cuda", generator=g)
    q = torch.rand(100, 2, device="cuda", generator=g) * 240
    a = tp.track(images, q[None], coarse_iters=2)
    out = tp.track_batch(images, [q], coarse_iters=2)
    b = cb.split_batch(out)[0]
    assert set(a) == set(b)
    for k in a:
        if isinstance(a[k], list):
            assert all(torch.equal(x, y) for x, y in zip(a[k], b[k])), k
        elif a[k] is None:
            assert b[k] is None
        else:
            assert torch.equal(a[k], b[k]), k


@pytest.mark.gpu
def test_track_batch_ragged_from_images(no_tf32):
    import comet_pose_estimation_b200 as cb

    tp = _tracker()
    g = torch.Generator(device="cuda").manual_seed(6)
    images = torch.randn(3, 4, 3, 256, 256, device="cuda", generator=g)
    with torch.no_grad():
        fm = tp._encode_frames(images)
        for b in range(3):
            # not bitwise: cuDNN may pick another convolution algorithm for B*S frames (1.03e-5 measured here)
            assert rel_to_max(fm[b:b + 1].cpu(), tp.process_images_to_fmaps(images[b:b + 1]).cpu()) < 2e-5
    qs = [torch.rand(n, 2, device="cuda", generator=g) * 240 for n in (90, 7, 200)]
    out = tp.track_batch(images, qs, coarse_iters=2)
    parts = cb.split_batch(out)
    for b, (p, q) in enumerate(zip(parts, qs)):
        one = tp.track(images[b:b + 1], q[None], coarse_iters=2)
        assert rel_to_max(p["coarse_pred_track_list"][0].cpu(), one["coarse_pred_track_list"][0].cpu()) < 1e-5, b
        for k, v in out.items():
            if isinstance(v, torch.Tensor) and v.dim() >= 3:
                assert torch.isfinite(v).all(), k
                assert torch.count_nonzero(v[b, :, q.shape[0]:]) == 0, k
