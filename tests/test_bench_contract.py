"""CPU-side checks of bench.py: the byte accounting behind `roofline`, the synthetic input layouts, and the JSON line
of the reference arm (`--impl reference` runs the CPU port, so it runs here)."""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def test_token_widths_and_algorithmic_bytes():
    assert bench.tdim(5, 4, 128, False) == 664 and bench.tdim(3, 3, 32, True) == 216   # base_track_predictor.py:55-66
    ab = bench.algorithmic_bytes(4, fine_layout="cl")
    # upper bound (every box fully inside its map): 23.7 KB per fine query, 8192 queries per sequence
    per_query = ab["fine_tokens"] / (4 * 512 * 16)
    assert abs(per_query - ((64 + 64 + 49) * 128 + 128 + 8 + 864 + 54)) < 1.0
    # SURVEY 8(d): 59.6 MB per coarse sequence-iteration
    assert abs(ab["coarse_tokens"] / 4 / 1e6 - 59.6) < 0.1
    assert ab["fine_pyramid"] == 4 * 512 * 16 * 32 * 4 * (900 + 225 + 49)
    up = bench.algorithmic_bytes(4, fine_layout="up2")
    assert abs(up["fine_tokens"] / (4 * 512 * 16) - ((81 + 49) * 128 + 128 + 8 + 864 + 54)) < 1.0
    assert up["fine_pyramid"] == 4 * 512 * 16 * 32 * 4 * (225 + 49)


def test_fine_bytes_are_clipped_to_the_maps_per_query():
    """VERDICT r1: taps off the map are zero padding the TMA unit never fetches; the algorithmic bytes count, per query,
    only the part of each box that lies on its map."""
    c = torch.tensor([[15.0, 15.0]])                       # centre: every box inside
    assert bench.fine_lines_per_query(c, "cl") == 64 + 64 + 49
    assert bench.fine_lines_per_query(c, "up2") == 81 + 49
    c = torch.tensor([[0.0, 0.0]])                         # corner: level 0 sees 5x5 of its 8x8 box, ...
    assert bench.fine_lines_per_query(c, "cl") == 5 * 5 + 5 * 5 + 5 * 5
    assert bench.fine_lines_per_query(c, "up2") == 6 * 6 + 5 * 5
    c = torch.tensor([[-100.0, 3.0]])                      # off the map: nothing to read
    assert bench.fine_lines_per_query(c, "cl") == 0 and bench.fine_lines_per_query(c, "up2") == 0
    d = bench.make_inputs(1, 3, torch, pin=False, fine_layout="up2")
    clipped = bench.algorithmic_bytes(1, d["fine"]["coords"], "up2")["fine_tokens"]
    assert clipped < bench.algorithmic_bytes(1, None, "up2")["fine_tokens"]


def test_synthetic_inputs_layouts():
    saved = dict(bench.FINE), dict(bench.COARSE)
    try:
        bench.FINE.update(P=3, S=2)
        bench.COARSE.update(S=2, N=5, H=8, W=8, C=4)
        ref = None
        for layout in ("up2", "cl", "nchw"):
            d = bench.make_inputs(2, 7, torch, pin=False, fine_layout=layout)
            f = d["fine"]["fmaps"]
            assert f.shape == ((6, 2, 32, 16, 16) if layout == "up2" else (6, 2, 32, 31, 31))
            assert f.is_contiguous() == (layout == "nchw")
            assert f.permute(0, 1, 3, 4, 2).is_contiguous() == (layout != "nchw")
            if layout == "up2":
                ref = bench.upsample_fine(torch, f, "nchw")
            else:
                assert torch.equal(f, ref)               # every layout carries the same values
            assert d["coarse"]["fmaps"].is_contiguous()
            c = d["fine"]["coords"]
            assert c.shape == (6, 6, 2, 1, 2)
            assert torch.equal(c[0][:, 0], c[5][:, 0])      # frame 0 stays pinned to the query point
    finally:
        bench.FINE.clear(); bench.FINE.update(saved[0])
        bench.COARSE.clear(); bench.COARSE.update(saved[1])


def test_dumped_outputs_are_a_fixed_sample_within_64_mb():
    rows = 4 * 512 * 16
    coarse = torch.arange(rows, dtype=torch.float32)[:, None].repeat(1, 664).reshape(4, 512, 16, 664)   # row i holds i
    fine = torch.randn(4 * 512, 1, 16, 216)
    a = bench.sample_outputs({"coarse_tokens": coarse, "fine_tokens": fine})
    b = bench.sample_outputs({"coarse_tokens": coarse, "fine_tokens": fine})
    assert sum(v.nbytes for v in a.values()) <= 64 * 10 ** 6
    assert a["fine_tokens"].dtype == np.float32 and np.array_equal(a["fine_tokens"], fine.numpy())   # fits: whole
    got = a["coarse_tokens"]
    assert got.shape[1] == 664 and 0 < got.shape[0] < rows and np.array_equal(got, b["coarse_tokens"])
    assert (got == got[:, :1]).all() and (np.diff(got[:, 0]) > 0).all()     # whole rows, distinct, in order


def test_reference_arm_json_line():
    env = dict(os.environ, OMP_NUM_THREADS="4")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--batch", "1"],
                       capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == bench.METRIC and line["unit"] == bench.UNIT
    assert line["higher_is_better"] is True and line["value"] > 0 and line["steps"] == 1
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"] == {"value": line["value"], "unit": bench.UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["gpu_launches"] == 0
    # both arms describe the workload with the same `config` (the driver's same_config check)
    assert line["config"] == bench.make_config(1, 1, "up2")
