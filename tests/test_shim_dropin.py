"""The C++/LibTorch drop-in, end to end inside the reference: oracle/_ref/ref_driver_b200 is the reference's OWN program
(unmodified sources: GlobalDataPool, Dataset, Renderer class, factories, autograd, loss) with the B200 code linked in at one
of two levels (INTEGRATION.md):

  fused  (default)    the body of Renderer::Render is f2nerf_b200/shim/B200Renderer.cpp — the fused C++ host of the hot path,
                      working on the reference's own PersSampler / Hash3DAnchored / SHShader objects;
  ops    (F2B_SHIM=ops)  the reference's own Renderer::Render drives the operator subclasses of shim/B200Ops.cpp.

oracle/_ref/ref_driver is the same program with nothing replaced.  All three run the same seeded script (512 ngp_fox rays),
so their dumps must agree: integer outputs and the sampler's fp32 outputs bit-exact, fp16-MLP-fed outputs within fp16 noise
of tiny-cuda-nn, gradients by cosine.  The fused C++ host must also equal the Python host mirror (f2nerf_b200/renderer.py)
bit for bit on every deterministic output: the two are the same kernel sequence.  The binaries are built only from the
reference's sources (build()); where they are absent, the C++ host's side of that last comparison is its committed record
tests/golden/shim_fused_512.npz (oracle/make_golden.py).
"""
import os
import subprocess
import tempfile

import numpy as np
import pytest
import torch

from test_gpu_parity import N, T
from test_ref_parity import build_from_ref, diag_path, kept_rows, load_record

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "oracle", "_ref", "ref_driver")
B200 = os.path.join(ROOT, "oracle", "_ref", "ref_driver_b200")
FUSED_RECORD = os.path.join(ROOT, "tests", "golden", "shim_fused_512.npz")
N_RAYS = 512
_runs = {}


def _run(kind):
    if kind in _runs:
        return _runs[kind]
    binary = REF if kind == "ref" else B200
    if not os.path.exists(binary):
        pytest.skip(f"{binary} not built (build() makes it from the reference's sources)")
    out = tempfile.mkdtemp(prefix=f"f2b_shim_{kind}_")
    env = dict(os.environ)
    env.pop("F2B_SHIM", None); env.pop("F2B_RENDER", None)
    if kind == "ops":
        env["F2B_SHIM"] = "ops"
    r = subprocess.run([binary, os.path.join(ROOT, "oracle", "ref_config_ngp_fox.yaml"), out, str(N_RAYS), "0", "1"],
                       cwd=ROOT, capture_output=True, text=True, timeout=900, env=env)
    open(diag_path(f"shim_{kind}.log"), "w").write(r.stdout[-8000:] + "\n--- stderr ---\n" + r.stderr[-8000:])
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    if kind == "ops":
        assert "replaced by the B200 subclasses" in r.stdout
    if kind == "fused":
        assert "replaced by the fused B200 host" in r.stdout
    _runs[kind] = {f[:-4]: np.load(os.path.join(out, f)) for f in os.listdir(out) if f.endswith(".npy")}
    return _runs[kind]


@pytest.fixture(params=["fused", "ops"])
def pair(request):
    return _run("ref"), _run(request.param), request.param


def cos(a, b):
    a, b = np.asarray(a, np.float64).reshape(-1), np.asarray(b, np.float64).reshape(-1)
    return float((a * b).sum() / (np.linalg.norm(a) * np.linalg.norm(b) + 1e-300))


def _node_fields(blob):
    """TreeNode blob -> the meaningful fields only (the reference never initialises the struct padding)."""
    t = np.ascontiguousarray(blob).view(np.uint8).reshape(-1, 64)
    return np.concatenate([t[:, :53], t[:, 56:60]], 1)


def test_same_scene(pair):
    a, b, _ = pair
    np.testing.assert_array_equal(_node_fields(a["tree_nodes"]), _node_fields(b["tree_nodes"]))
    for k in ("pers_trans", "edge_pool", "prim_pool", "bias_pool", "field_mlp_params", "shader_mlp_params", "app_emb",
              "rays_o", "rays_d", "train_noise", "train_bg", "train_edge_idx", "train_edge_coord"):
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)


def test_sampler_through_reference_program(pair):
    a, b, _ = pair
    for k in ("val_bounds", "val_anchors", "train_bounds", "train_anchors", "edge_anchors"):
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    for k in ("val_pts", "val_dt", "val_t", "val_first_oct_dis", "train_pts", "train_dt", "train_t", "train_first_oct_dis", "edge_pts"):
        np.testing.assert_array_equal(a[k].view(np.uint32), b[k].view(np.uint32), err_msg=k)


def test_render_through_reference_program(pair):
    a, b, kind = pair
    for mode in ("val", "train"):
        ca, cb = a[f"{mode}_idx_start_end"], b[f"{mode}_idx_start_end"]
        na, nb = ca[:, 1] - ca[:, 0], cb[:, 1] - cb[:, 0]
        # the T > 1e-4 crossing sits downstream of the fp16 MLP: tcnn's fp16-accumulate noise shifts it by a few samples
        assert (na == nb).mean() >= 0.9 and abs(int(na.sum()) - int(nb.sum())) <= 2e-3 * na.sum(), (mode, (na == nb).mean())
        np.testing.assert_allclose(b[f"{mode}_colors"], a[f"{mode}_colors"], atol=0.03, err_msg=mode)        # fp16 MLP outputs, composited
        assert np.median(np.abs(b[f"{mode}_colors"] - a[f"{mode}_colors"])) <= 3e-3
        for k in ("depth", "disparity"):
            rel = np.abs(b[f"{mode}_{k}"] - a[f"{mode}_{k}"]) / (np.abs(a[f"{mode}_{k}"]) + 1e-3)
            assert np.median(rel) <= 1e-2, (mode, k, np.median(rel))
    assert abs(float(b["train_loss"][0]) - float(a["train_loss"][0])) <= 5e-3 * abs(float(a["train_loss"][0]))
    assert a["backward_nan"][0] == 0 and b["backward_nan"][0] == 0
    # octree occupancy state after UpdateOctNodes: votes depend on the (fp16-noisy) early weights through thresholds
    for k in ("train_weight_stats_after", "train_alpha_stats_after", "train_visit_cnt_after"):
        assert (a[k] != b[k]).mean() <= 2e-3, k
    assert (_node_fields(a["train_tree_nodes_after"]) != _node_fields(b["train_tree_nodes_after"])).mean() <= 1e-4
    ef_a, ef_b = a["train_edge_feats"], b["train_edge_feats"]
    assert cos(ef_a, ef_b) >= 0.999
    for name in ("grad_field_mlp", "grad_shader_mlp", "grad_app_emb"):
        assert cos(a[name], b[name]) >= 0.98, (kind, name, cos(a[name], b[name]))
    assert cos(a["grad_feat_pool"], b["grad_feat_pool"]) >= 0.97, (kind, cos(a["grad_feat_pool"], b["grad_feat_pool"]))


def test_fused_cpp_host_equals_python_host():
    """B200Renderer.cpp and f2nerf_b200/renderer.py are the same kernel sequence: every deterministic output of the seeded
    TRAIN step is bit-identical; the atomically accumulated gradients agree to fp32 summation order."""
    from f2nerf_b200 import TRAIN, CustomOps, check_backward_nan
    c = _run("fused") if os.path.exists(B200) else load_record(FUSED_RECORD)
    gdp, sampler, field, shader, renderer = build_from_ref(c)
    gdp.mode_, gdp.iter_step_, gdp.ray_march_fineness_, gdp.gradient_scaling_progress_ = TRAIN, 1, 1.0, 0.25
    rays_o, rays_d, emb_idx, gt = T(c["rays_o"]), T(c["rays_d"]), T(c["emb_idx"]), T(c["gt_colors"])
    torch.manual_seed(777)
    r = renderer.Render(rays_o, rays_d, None, emb_idx)
    loss = (torch.sqrt((r.colors - gt) ** 2 + 1e-4).mean() + torch.sqrt(CustomOps.WeightVar(r.weights, r.idx_start_end) + 1e-2).mean() * 1e-2
            + (r.disparity ** 2).mean() * 1e-2 + ((r.edge_feats[:, 0] - r.edge_feats[:, 1]) ** 2).mean() * 1e-1)
    loss.backward()
    assert not check_backward_nan(renderer)
    np.testing.assert_array_equal(N(r.idx_start_end), c["train_idx_start_end"])
    for k, v in (("train_colors", r.colors), ("train_disparity", r.disparity), ("train_depth", r.depth), ("train_weights", r.weights),
                 ("train_edge_feats", r.edge_feats), ("train_first_oct_dis", r.first_oct_dis)):
        np.testing.assert_array_equal(kept_rows(c, k + "_idx", N(v)).view(np.uint32), c[k].view(np.uint32), err_msg=k)
    for k, v in (("train_weight_stats_after", sampler.tree_weight_stats_), ("train_alpha_stats_after", sampler.tree_alpha_stats_),
                 ("train_visit_cnt_after", sampler.tree_visit_cnt_)):
        np.testing.assert_array_equal(N(v).reshape(-1), c[k].reshape(-1), err_msg=k)
    np.testing.assert_array_equal(_node_fields(N(sampler.tree_nodes_gpu_)), _node_fields(c["train_tree_nodes_after"]))
    assert abs(float(loss) - float(c["train_loss"][0])) <= 1e-6 * abs(float(loss))
    table = (field.feat_pool_.grad, c["grad_feat_pool"]) if "grad_feat_pool" in c else \
        (field.feat_pool_.grad.reshape(-1)[torch.from_numpy(c["grad_feat_pool_sub_idx"]).cuda()], c["grad_feat_pool_sub_val"])
    for name, g, want in (("grad_field_mlp", field.mlp_.params_.grad, c["grad_field_mlp"]),
                          ("grad_shader_mlp", shader.mlp_.params_.grad, c["grad_shader_mlp"]),
                          ("grad_app_emb", renderer.app_emb_.grad, c["grad_app_emb"]), ("grad_feat_pool",) + table):
        a, b = N(g).astype(np.float64).reshape(-1), want.astype(np.float64).reshape(-1)
        assert np.linalg.norm(a - b) <= 1e-5 * np.linalg.norm(b), (name, np.linalg.norm(a - b) / np.linalg.norm(b))
