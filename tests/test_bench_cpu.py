"""Host-side logic of bench.py that must not break on the GPU box (no GPU needed): the `config` object both arms print, the governing
rooflines computed from the committed captures / microbenchmarks, the clock sampler on ranks that do not sample, the arrays
--dump-outputs writes."""
import glob
import json
import os
import sys
from types import SimpleNamespace

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
import workloads as W  # noqa: E402


def test_config_object_is_a_pure_function_of_the_flags():
    for cfg in sorted(W.CONFIGS):
        a = bench.config_dict(SimpleNamespace(config=cfg, rays=0), 1)
        b = bench.config_dict(SimpleNamespace(config=cfg, rays=0), 1)
        assert a == b and a["name"] == cfg and "workload" in a and "model" not in a
    strong = bench.config_dict(SimpleNamespace(config="nerf360", rays=0), 8)
    assert strong["rays_per_gpu"] * 8 == strong["global_rays"] == 8192                       # one global batch, split
    weak = bench.config_dict(SimpleNamespace(config="wanjinyou", rays=0), 8)
    assert weak["rays_per_gpu"] == 4096 and weak["global_rays"] == 8 * 4096


def test_governing_rooflines_from_committed_profiles():
    """profiles/*_traffic.json (ncu sector counts) + the two microbenchmark files must give sane fractions for the two table
    kernels at their measured times, and nothing for kernels / workloads they do not describe."""
    assert glob.glob(os.path.join(ROOT, "profiles", "*_traffic.json"))
    bench.GOVERNING_OK = True
    g = bench.governing_roofline("f2b_field_fwd_slots", 0.90)
    assert g["bound"] == "l1_l2_gather_sectors" and 0.9 < g["frac"] <= 1.01 and g["units_per_launch"] > 2e8
    r = bench.governing_roofline("f2b_hash_bwd", 0.87)
    assert r["bound"] == "l2_reduction_issue" and 0.6 < r["frac"] < 0.95 and r["units_per_launch"] > 1e8
    assert bench.governing_roofline("f2b_composite_fwd", 0.1) is None
    bench.GOVERNING_OK = False                                                                # any other workload than the captured one
    assert bench.governing_roofline("f2b_hash_bwd", 0.87) is None
    bench.GOVERNING_OK = True
    t = bench.ncu_traffic("f2b_hash_bwd")
    assert t is not None and t["dram_bytes_per_launch"] > 1e8


def test_clock_sampler_is_inert_on_non_sampling_ranks():
    c = bench.ClockSampler(-1)
    c.poll()
    assert c.rows == [] and "not sampled" in c.err
    s = c.summary()
    assert s["sm_mhz"] is None


def test_committed_bench_lines_carry_the_contract_keys():
    """The driver-format lines kept under profiles/ (the numbers DESIGN.md / BASELINE.md quote) have every key of the bench contract."""
    line = json.loads(open(os.path.join(ROOT, "profiles", "r02q_bench.json")).read().strip().splitlines()[-1])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
              "data", "config", "e2e", "gpu_launches", "clocks", "roofline", "cpu_baseline"):
        assert k in line, k
    assert line["vs_baseline"] is None and line["roofline"]["bound"] in ("hbm", "tensor") and line["gpu_launches"] > 0
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(line["e2e"])
    assert {"value", "unit", "cores", "kind", "sample"} <= set(line["cpu_baseline"])
    ref = json.loads(open(os.path.join(ROOT, "profiles", "r02h_bench_ref.json")).read().strip().splitlines()[-1])
    assert ref["impl"] == "reference" and ref["config"] == line["config"] and ref["metric"] == line["metric"]
    gov = {r["kernel"]: r["governing"] for r in line["rooflines"]}
    assert 0.9 < gov["f2b_field_fwd_slots"]["frac"] <= 1.01 and 0.6 < gov["f2b_hash_bwd"]["frac"] < 0.95


def test_dump_outputs_types_sampling_and_files(tmp_path):
    """Every returned array becomes DIR/<name>.npy in float32 (integers in float64); one larger than DUMP_CAP is replaced by the
    same seeded sample of its elements on every call."""
    grad = lambda *shape: SimpleNamespace(grad=torch.rand(shape))
    table = torch.rand(bench.DUMP_CAP + 5, 2)
    prob = dict(field=SimpleNamespace(feat_pool_=SimpleNamespace(grad=table), mlp_=SimpleNamespace(params_=grad(8))),
                shader=SimpleNamespace(mlp_=SimpleNamespace(params_=grad(4))), renderer=SimpleNamespace(app_emb_=SimpleNamespace(grad=None)))
    res = SimpleNamespace(colors=torch.rand(6, 3), disparity=torch.rand(6), depth=torch.rand(6), first_oct_dis=torch.rand(6, 1),
                          weights=torch.rand(20), idx_start_end=torch.arange(12, dtype=torch.int32).reshape(6, 2),
                          edge_feats=torch.rand(4, 2, 16))
    out = bench.step_outputs(prob, torch.tensor(0.5, requires_grad=True), res)
    assert "grad_app_emb" not in out and out["loss"].shape == (1,) and out["colors"].shape == (6, 3)
    assert out["idx_start_end"].dtype == np.float64 and (out["idx_start_end"] == np.arange(12).reshape(6, 2)).all()
    assert all(a.dtype == np.float32 for k, a in out.items() if k != "idx_start_end")
    assert out["grad_feat_pool"].shape == (bench.DUMP_CAP,) and np.isin(out["grad_feat_pool"][:100], table.numpy()).all()
    np.testing.assert_array_equal(out["grad_feat_pool"], bench.step_outputs(prob, torch.tensor(0.5), res)["grad_feat_pool"])
    bench.write_outputs(str(tmp_path / "d"), out)
    assert sorted(os.listdir(tmp_path / "d")) == sorted(k + ".npy" for k in out)
    np.testing.assert_array_equal(np.load(tmp_path / "d" / "weights.npy"), out["weights"])
