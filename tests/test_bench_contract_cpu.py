"""bench.py's contract pieces that need no GPU: the algorithmic-FLOP model (SURVEY.md 8d), the `config` object shared by both
arms, the roofline denominators and the ncu traffic lookup from the committed summary."""
import importlib.util
import json
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]


@pytest.fixture(scope="module")
def bench():
    spec = importlib.util.spec_from_file_location("bench_module", ROOT / "bench.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_algorithmic_flops_per_view_match_the_survey(bench):
    # SURVEY.md 8(d): totals per view 2.03 T (V=2), 2.45 T (V=8), 3.55 T (V=24), 8.80 T (V=100), 71.0 T (V=1000)
    for v, want in ((2, 2.03), (8, 2.45), (24, 3.55), (100, 8.80), (1000, 71.0)):
        assert abs(bench.gflop_per_view(v) / 1e3 - want) < 0.02 * want, (v, bench.gflop_per_view(v))


def test_config_object_is_shared_by_both_arms_and_names_the_baseline_config(bench):
    c1 = bench.bench_config(8, 1, "shard", False, False)
    assert c1 == bench.bench_config(8, 1, "shard", False, False)
    assert c1["views"] == 8 and c1["scene_views"] == 8 and c1["parallelism"] == "single" and "model" not in c1
    assert "8 views" in c1["workload"] and "config[1]" in c1["workload"]
    c8 = bench.bench_config(8, 8, "shard", False, True)
    assert c8["views"] == 64 and c8["scene_views"] == 64 and "all-gather" in c8["parallelism"]
    assert abs(c8["tflop_per_view"] - bench.gflop_per_view(64) / 1e3) < 1e-9
    rep = bench.bench_config(8, 4, "replicas", False, False)
    assert rep["scene_views"] == 8 and rep["views"] == 32 and rep["parallelism"] == "replicas x4"
    mm = bench.bench_config(24, 1, "shard", True, False)
    assert "multi-modal" in mm["workload"] and "config[2]" in mm["workload"]
    json.dumps(c8)   # plain JSON


def test_roofline_denominators_and_traffic_lookup(bench):
    tf, hbm, src = bench.measured_peaks()
    assert src in ("measured", "fallback") and 1000 < tf < 2300 and 5000 < hbm < 8100
    traffic, note = bench.ncu_gemm_traffic()
    # the committed ncu summary of the dominant GEMM launch: within 1.5x of its algorithmic 120.6 MB
    assert traffic is not None and 0.5 * 120.6e6 < traffic < 1.5 * 120.6e6, (traffic, note)
    assert "profiles/" in note


def test_dump_outputs_fits_the_budget_with_a_fixed_pixel_sample(bench, tmp_path):
    """--dump-outputs on the forward() dicts of 5 views at 518 px (70 MB of outputs): float32 files within the budget, the
    same seeded pixel sample for every view and key, per-view vectors whole, identical from run to run."""
    import numpy as np
    import torch

    V, S = 5, bench.IMG
    P = S * S

    def view(i):
        px = (torch.arange(P, dtype=torch.float32) + i * P).view(1, S, S)   # every value names its view and pixel
        return {"pts3d": px[..., None].repeat(1, 1, 1, 3), "pts3d_cam": px[..., None].repeat(1, 1, 1, 3),
                "ray_directions": px[..., None].repeat(1, 1, 1, 3), "depth_along_ray": px[..., None], "conf": px.clone(),
                "non_ambiguous_mask_logits": -px, "non_ambiguous_mask": px % 2 == 1,
                "cam_trans": torch.full((1, 3), float(i)), "cam_quats": torch.full((1, 4), float(i)),
                "metric_scaling_factor": torch.ones(1, 1)}

    preds = [view(i) for i in range(V)]
    bench.dump_outputs(preds, str(tmp_path / "a"))
    bench.dump_outputs(preds, str(tmp_path / "b"))
    got = {f.stem: np.load(f) for f in (tmp_path / "a").glob("*.npy")}
    assert set(got) == set(preds[0])
    assert all(a.dtype == np.float32 for a in got.values())
    assert 0.95 * bench.DUMP_BYTES < sum(a.nbytes for a in got.values()) <= bench.DUMP_BYTES
    for k, a in got.items():
        assert np.array_equal(a, np.load(tmp_path / "b" / f"{k}.npy")), k
    assert np.array_equal(got["cam_quats"], np.repeat(np.arange(V, dtype=np.float32)[:, None], 4, 1))
    assert got["metric_scaling_factor"].shape == (V, 1)
    pix = got["conf"][0]
    n = pix.size
    assert 0 < n < P and np.all(np.diff(pix) > 0)
    for i in range(V):
        assert np.array_equal(got["conf"][i], pix + i * P)
        assert np.array_equal(got["pts3d"][i], np.repeat((pix + i * P)[:, None], 3, 1))
        assert np.array_equal(got["non_ambiguous_mask"][i], (pix + i * P) % 2)
    assert got["depth_along_ray"].shape == (V, n, 1)
