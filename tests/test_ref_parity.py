"""CUDA path against the REAL reference (unmodified Totoro97/f2-nerf + tiny-cuda-nn, compiled into
oracle/_ref/ref_driver) on the reference's own ngp_fox octree / cameras, from two sources:

  * ``golden`` — the committed dump of a 40-ray reference run, tests/golden/ref_ngp_fox.npz (oracle/make_golden.py);
  * ``live``   — the reference run at 512 rays: the binary on this GPU where it is built (oracle/_ref/ref_driver, made by
    build() from the reference's sources), otherwise its committed record tests/golden/ref_ngp_fox_512.npz
    (oracle/make_golden.py), which keeps every per-ray output and seeded samples of the per-sample ones.

Integer outputs (sample bounds, anchors, compacted bounds, octree statistics and pruned nodes) must be
bit-exact; fp32 stages within 1e-4; fp16 stages (hash features -> tcnn MLP) within fp16 noise of tcnn.
"""
import json
import os
import subprocess
import tempfile

import numpy as np
import pytest
import torch

from test_gpu_parity import N, T, assert_close, half_ulps

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DRV = os.path.join(ROOT, "oracle", "_ref", "ref_driver")
N_RAYS_LIVE = 512
GOLD = os.path.join(ROOT, "tests", "golden", "ref_ngp_fox.npz")
LIVE_RECORD = os.path.join(ROOT, "tests", "golden", "ref_ngp_fox_512.npz")
BOTH = ["golden", "live"]


def diag_path(name):
    """Where a test leaves its JSON / log diagnostics: $F2B_DIAG_DIR, else a per-user directory under the system temp dir."""
    d = os.environ.get("F2B_DIAG_DIR") or os.path.join(tempfile.gettempdir(), f"f2b_diag_{os.getuid()}")
    os.makedirs(d, exist_ok=True)
    return os.path.join(d, name)


def load_record(path):
    """A committed record of a 512-ray run (oracle/make_golden.py); the entries it shares with the 40-ray fixture live there."""
    d = dict(np.load(path))
    gold = np.load(GOLD)
    for k in d.pop("from_ref_ngp_fox"):
        d[str(k)] = gold[str(k)]
    return d


def kept_rows(ref, idx_key, a):
    """``a`` (ours, every row) restricted to the rows a committed record keeps (``ref[idx_key]``); a full dump keeps them all."""
    return a[ref[idx_key]] if idx_key in ref else a


def _live():
    if not os.path.exists(DRV):
        return load_record(LIVE_RECORD)
    out = tempfile.mkdtemp(prefix="f2b_ref_dump_")              # large (full 64 MB table gradient)
    r = subprocess.run([DRV, os.path.join(ROOT, "oracle", "ref_config_ngp_fox.yaml"), out, str(N_RAYS_LIVE), "0", "1"], cwd=ROOT,
                       capture_output=True, text=True, timeout=900)
    open(diag_path("ref_driver.log"), "w").write(r.stdout[-20000:] + "\n--- stderr ---\n" + r.stderr[-20000:])
    assert r.returncode == 0, r.stderr[-3000:]
    return {f[:-4]: np.load(os.path.join(out, f)) for f in os.listdir(out) if f.endswith(".npy")}


_cache = {}


@pytest.fixture(params=BOTH)
def ref(request):
    """The reference's dumps, keyed like ref_driver.cpp names them.  fp16-stored fixture entries are widened to fp32."""
    kind = request.param
    if kind not in _cache:
        d = _live() if kind == "live" else dict(np.load(GOLD))
        _cache[kind] = {k: (v.astype(np.float32) if v.dtype == np.float16 else v) for k, v in d.items()}
    d = _cache[kind]
    d["_kind"] = kind
    return d


def n_rays_of(ref):
    return int(ref["scalars"][7])


def build_from_ref(ref):
    from f2nerf_b200 import GlobalDataPool, Hash3DAnchored, PersSampler, Renderer, SHShader
    sc = ref["scalars"]
    near, sample_l, scale_by_dis, max_hits, V, pool, n_img = float(sc[0]), float(sc[1]), bool(sc[2]), int(sc[3]), int(sc[4]), int(sc[5]), int(sc[6])
    gdp = GlobalDataPool()
    sampler = PersSampler(gdp, ref["tree_nodes"], ref["pers_trans"], ref["edge_pool"], near=near, sample_l=sample_l,
                          scale_by_dis=scale_by_dis, max_oct_intersect_per_ray=max_hits)
    assert gdp.n_volumes_ == V
    log2 = int(np.log2(pool // 16))
    field = Hash3DAnchored(gdp, log2_table_size=log2, prim_pool=ref["prim_pool"], bias_pool=ref["bias_pool"])
    g = torch.Generator().manual_seed(1234)                       # same CPU generator stream as ref_driver.cpp
    field.feat_pool_.data.copy_((torch.rand((pool, 2), generator=g) * 2. - 1.).cuda())
    field.mlp_.params_.data.copy_(T(ref["field_mlp_params"]))
    shader = SHShader(gdp)
    shader.mlp_.params_.data.copy_(T(ref["shader_mlp_params"]))
    renderer = Renderer(gdp, sampler, field, shader, n_images=n_img, use_app_emb=True)
    renderer.app_emb_.data.copy_((torch.rand((n_img, 16), generator=g) * .2 - .1).cuda())
    np.testing.assert_array_equal(N(renderer.app_emb_), ref["app_emb"])
    return gdp, sampler, field, shader, renderer


def test_mlp_init_matches_tcnn(ref):
    """pcg32 xavier init: our host-side stream vs tiny-cuda-nn's initialize_params (x4 for the field)."""
    from f2nerf_b200.field import tcnn_xavier_params
    np.testing.assert_array_equal(tcnn_xavier_params(32, 2).numpy(), ref["shader_mlp_params"])
    np.testing.assert_array_equal(tcnn_xavier_params(32, 1).numpy() * 4.0, ref["field_mlp_params"])


def test_sampler_validate_bit_exact(ref):
    from f2nerf_b200 import VALIDATE
    gdp, sampler, field, shader, renderer = build_from_ref(ref)
    gdp.mode_ = VALIDATE
    s = sampler.GetSamples(T(ref["rays_o"]), T(ref["rays_d"]), None)
    np.testing.assert_array_equal(N(s.pts_idx_bounds), ref["val_bounds"])
    np.testing.assert_array_equal(kept_rows(ref, "val_sample_idx", N(s.anchors)[:, :2]), ref["val_anchors"])
    np.testing.assert_array_equal(N(s.first_oct_dis).view(np.uint32), ref["val_first_oct_dis"].view(np.uint32))
    for k, v in (("val_t", s.t), ("val_dt", s.dt), ("val_dirs", s.dirs), ("val_pts", s.pts)):
        np.testing.assert_array_equal(kept_rows(ref, "val_sample_idx", N(v)).view(np.uint32), ref[k].view(np.uint32), err_msg=k)


def test_field_and_shader_vs_tcnn(ref):
    from f2nerf_b200 import VALIDATE
    gdp, sampler, field, shader, renderer = build_from_ref(ref)
    gdp.mode_ = VALIDATE
    with torch.no_grad():
        pts, anchors, dirs = T(ref["val_pts"]), T(np.ascontiguousarray(ref["val_anchors"][:, 0])), T(ref["val_dirs"])
        feat = field.AnchoredQuery(pts, anchors)
        # tcnn accumulates in fp16 inside wmma: compare at fp16 resolution of the output scale
        scale = np.abs(ref["val_scene_feat"]).max()
        err = np.abs(N(feat) - ref["val_scene_feat"])
        assert err.max() <= 0.02 * scale and np.median(err) <= 2e-3 * scale, (err.max(), np.median(err), scale)
        shading = torch.cat([torch.ones_like(feat[:, :1]), T(ref["val_scene_feat"])[:, 1:]], 1)
        rgb = shader.Query(shading, dirs)
        assert np.abs(N(rgb) - ref["val_rgb"]).max() <= 0.02


def test_render_validate_vs_reference(ref):
    from f2nerf_b200 import VALIDATE
    gdp, sampler, field, shader, renderer = build_from_ref(ref)
    gdp.mode_ = VALIDATE
    with torch.no_grad():
        r = renderer.Render(T(ref["rays_o"]), T(ref["rays_d"]), None, None)
    same_mask = np.array_equal(N(r.idx_start_end), ref["val_idx_start_end"])
    mine, theirs = N(r.idx_start_end), ref["val_idx_start_end"]
    cnt_m, cnt_t = mine[:, 1] - mine[:, 0], theirs[:, 1] - theirs[:, 0]
    frac_rays_same = (cnt_m == cnt_t).mean()
    json.dump(dict(frac_rays_same_count=float(frac_rays_same), max_count_diff=int(np.abs(cnt_m - cnt_t).max()),
                   kept_mine=int(cnt_m.sum()), kept_ref=int(cnt_t.sum())), open(diag_path("ref_validate_mask.json"), "w"))
    # the T > 1e-4 crossing sits downstream of the fp16 MLP: tcnn's fp16-accumulate noise shifts it by a few samples
    assert frac_rays_same >= 0.9 and abs(int(cnt_m.sum()) - int(cnt_t.sum())) <= 2e-3 * cnt_t.sum(), (frac_rays_same, cnt_m.sum(), cnt_t.sum())
    assert np.abs(N(r.colors) - ref["val_colors"]).max() <= 0.03
    assert np.median(np.abs(N(r.colors) - ref["val_colors"])) <= 3e-3
    assert np.median(np.abs(N(r.depth) - ref["val_depth"]) / (np.abs(ref["val_depth"]) + 1e-3)) <= 1e-2
    if same_mask:
        assert np.median(np.abs(kept_rows(ref, "val_weights_idx", N(r.weights)) - ref["val_weights"])) <= 1e-3


def test_edge_samples_vs_reference(ref):
    """PersSampler::GetEdgeSamples: the kernel on the reference's own draws, and the seeded draws themselves."""
    from f2nerf_b200 import ops
    gdp, sampler, field, shader, renderer = build_from_ref(ref)
    pts, idx = ops.edge_samples(sampler.edge_pool_gpu_, sampler.pers_trans_gpu_, T(ref["edge_idx"]), T(ref["edge_coord"]))
    np.testing.assert_array_equal(N(idx), ref["edge_anchors"])
    diff = np.abs(N(pts).astype(np.float64) - ref["edge_pts"].astype(np.float64))
    json.dump(dict(max_abs=float(diff.max()), frac_bit_exact=float((N(pts).view(np.uint32) == ref["edge_pts"].view(np.uint32)).mean())),
              open(diag_path("ref_edge_samples.json"), "w"))
    np.testing.assert_array_equal(N(pts).view(np.uint32), ref["edge_pts"].view(np.uint32))       # bit-exact
    torch.manual_seed(4242)                                       # same Philox stream => identical draws through our mirror
    e_pts, e_idx = sampler.GetEdgeSamples(8192)
    n = ref["edge_anchors"].shape[0]                              # the committed fixture keeps the first 2048 of the 8192 draws
    np.testing.assert_array_equal(N(e_idx)[:n], ref["edge_anchors"])
    np.testing.assert_array_equal(N(e_pts)[:n].view(np.uint32), ref["edge_pts"].view(np.uint32))


def test_render_train_vs_reference(ref):
    """Seeded TRAIN-mode step: same torch RNG draws, octree votes bit-exact, gradients close."""
    from f2nerf_b200 import TRAIN, CustomOps, check_backward_nan
    gdp, sampler, field, shader, renderer = build_from_ref(ref)
    gdp.mode_, gdp.iter_step_, gdp.ray_march_fineness_, gdp.gradient_scaling_progress_ = TRAIN, 1, 1.0, 0.25
    rays_o, rays_d, emb_idx, gt = T(ref["rays_o"]), T(ref["rays_d"]), T(ref["emb_idx"]), T(ref["gt_colors"])
    torch.manual_seed(777)
    noise = sampler.make_noise(n_rays_of(ref), rays_o.device)
    np.testing.assert_array_equal(N(noise), ref["train_noise"])           # same Philox stream as the reference run
    torch.manual_seed(777)
    r = renderer.Render(rays_o, rays_d, None, emb_idx)
    sr = renderer.sample_result_
    np.testing.assert_array_equal(N(sr.pts_idx_bounds), ref["train_bounds"])
    np.testing.assert_array_equal(kept_rows(ref, "train_sample_idx", N(sr.anchors)[:, :2]), ref["train_anchors"])
    for k, v in (("train_t", sr.t), ("train_dt", sr.dt), ("train_pts", sr.pts)):
        np.testing.assert_array_equal(kept_rows(ref, "train_sample_idx", N(v)).view(np.uint32), ref[k].view(np.uint32), err_msg=k)
    # octree occupancy state after UpdateOctNodes: votes depend on the (fp16-noisy) early weights through
    # thresholds, so allow a tiny number of flipped votes but require byte equality of everything else
    for mine, theirs in ((sampler.tree_weight_stats_, "train_weight_stats_after"), (sampler.tree_alpha_stats_, "train_alpha_stats_after"),
                         (sampler.tree_visit_cnt_, "train_visit_cnt_after")):
        assert (N(mine) != ref[theirs]).mean() <= 2e-3, theirs
    assert (N(sampler.tree_nodes_gpu_) != ref["train_tree_nodes_after"]).mean() <= 1e-4
    color_loss = torch.sqrt((r.colors - gt) ** 2 + 1e-4).mean()
    var_loss = torch.sqrt(CustomOps.WeightVar(r.weights, r.idx_start_end) + 1e-2).mean()
    tv = ((r.edge_feats[:, 0] - r.edge_feats[:, 1]) ** 2).mean()
    loss = color_loss + var_loss * 1e-2 + (r.disparity ** 2).mean() * 1e-2 + tv * 1e-1
    loss.backward()
    assert not check_backward_nan(renderer) and ref["backward_nan"][0] == 0
    assert abs(float(loss) - float(ref["train_loss"][0])) <= 5e-3 * abs(float(ref["train_loss"][0]))
    assert np.abs(N(r.colors) - ref["train_colors"]).max() <= 0.03
    summary = {}
    if "train_edge_feats" in ref:                     # same Philox draws => same edge points => same features (fp16 MLP noise)
        from f2nerf_b200 import ops as _ops
        from f2nerf_b200.field import field_forward
        n_e = ref["train_edge_feats"].shape[0]                   # fixture: first 2048 edge pairs
        ef_m, ef_t = N(r.edge_feats)[:n_e].astype(np.float64), ref["train_edge_feats"].astype(np.float64)
        cs = lambda a, b: float((a * b).sum() / (np.linalg.norm(a) * np.linalg.norm(b) + 1e-30))
        with torch.no_grad():                         # our field on the reference's replayed draws
            rp, ri = _ops.edge_samples(sampler.edge_pool_gpu_, sampler.pers_trans_gpu_, T(ref["train_edge_idx"][:n_e]),
                                       T(ref["train_edge_coord"][:n_e]))
            rep, _, _ = field_forward(field, field.table_f16(), field.mlp_.params_f16(), rp.reshape(-1, 3).contiguous(),
                                      ri.reshape(-1).contiguous(), 1, save=False)
        ef_r = N(rep).astype(np.float64).reshape(ef_t.shape)
        row_close = (np.abs(ef_m - ef_t).max(-1) <= 0.05 * (np.abs(ef_t).max(-1) + 1e-3))
        summary["edge_feats"] = dict(max_abs=float(np.abs(ef_m - ef_t).max()), ref_abs_max=float(np.abs(ef_t).max()),
                                     cos_ours_ref=cs(ef_m, ef_t), cos_ours_replay=cs(ef_m, ef_r), cos_replay_ref=cs(ef_r, ef_t),
                                     frac_rows_close=float(row_close.mean()), frac_rows_close_a=float(row_close[:, 0].mean()),
                                     frac_rows_close_b=float(row_close[:, 1].mean()),
                                     per_channel_cos=[cs(ef_m[..., k], ef_t[..., k]) for k in range(16)])
        json.dump(summary, open(diag_path("ref_edge_feats.json"), "w"), indent=1)
        # identical edge points (RNG-stream parity incl. the reference's torch::rand output buffers): fp16 MLP noise only
        assert summary["edge_feats"]["cos_ours_ref"] >= 0.999 and summary["edge_feats"]["frac_rows_close"] >= 0.97, summary["edge_feats"]
    if "grad_feat_pool" in ref:
        table_pair = (field.feat_pool_.grad.reshape(-1), ref["grad_feat_pool"])
    else:                                             # committed fixture: a seeded 2^18-element subsample of the live prefix
        sub = torch.from_numpy(ref["grad_feat_pool_sub_idx"]).cuda()
        table_pair = (field.feat_pool_.grad.reshape(-1)[sub], ref["grad_feat_pool_sub_val"])
    for name, mine, theirs in (("field_mlp", field.mlp_.params_.grad, ref["grad_field_mlp"]),
                               ("shader_mlp", shader.mlp_.params_.grad, ref["grad_shader_mlp"]),
                               ("app_emb", renderer.app_emb_.grad, ref["grad_app_emb"]),
                               ("feat_pool",) + table_pair):
        a, b = N(mine).astype(np.float64).reshape(-1), theirs.astype(np.float64).reshape(-1)
        cos = float((a * b).sum() / (np.linalg.norm(a) * np.linalg.norm(b) + 1e-30))
        rel = float(np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-30))
        summary[name] = dict(cos=cos, rel_l2=rel)
    if "grad_feat_pool" not in ref:
        S = field.local_size_
        mine_flat = field.feat_pool_.grad.reshape(-1).double()
        norms = np.array([float(torch.linalg.norm(mine_flat[l * S:(l + 1) * S])) for l in range(17)])
        summary["slab_norm_ratio"] = (norms / np.maximum(ref["grad_feat_pool_slab_norm"].astype(np.float64), 1e-30)).tolist()
        json.dump(summary, open(diag_path("golden_grad_parity.json"), "w"), indent=1)
        for name in ("field_mlp", "shader_mlp", "app_emb"):
            assert summary[name]["cos"] >= 0.98 and summary[name]["rel_l2"] <= 0.2, (name, summary[name])
        assert summary["feat_pool"]["cos"] >= 0.97, summary
        assert all(0.8 <= r <= 1.25 for r in summary["slab_norm_ratio"] if np.isfinite(r)), summary["slab_norm_ratio"]
        if ref["_kind"] == "golden":
            return
    # The reference rounds every (weight x grad*128) product of the hash scatter to fp16 before an fp16
    # atomicAdd (Hash3DAnchored.cu:145-151): tiny per-sample gradients underflow, so ITS table gradient is the
    # noisy side.  Emulating that rounding in the oracle (exact accumulation otherwise) must explain the gap.
    import oracle_pipeline as OP
    from f2nerf_b200 import ops
    sc = dict(nodes=ref["tree_nodes"], trans=ref["pers_trans"], edges=ref["edge_pool"], near=sampler.global_near_,
              sample_l=sampler.sample_l_, scale_by_dis=sampler.scale_by_dis_, max_hits=sampler.max_oct_intersect_per_ray_)
    fld = dict(table16=N(field.table_f16()), prim=N(field.prim_pool_), bias=N(field.bias_pool_), V=field.n_volumes_,
               local_size=field.local_size_, mlp_params=ref["field_mlp_params"])
    orc = OP.render_train(sc, ref["rays_o"], ref["rays_d_normed"], ref["train_noise"], ref["train_bg"], fld, ref["shader_mlp_params"],
                          ref["app_emb"], ref["emb_idx"], (ref["train_edge_idx"], ref["train_edge_coord"]), ref["gt_colors"],
                          scales=ops.hash_level_scales().numpy(), gs_progress=0.25, diagnostics="grad_feat_pool" in ref)
    def cosd(x, y):
        x, y = np.asarray(x, np.float64).reshape(-1), np.asarray(y, np.float64).reshape(-1)
        return float((x * y).sum() / (np.linalg.norm(x) * np.linalg.norm(y) + 1e-30))
    summary["feat_pool_ours_vs_oracle_exact"] = cosd(N(field.feat_pool_.grad), orc["grad_feat_pool"])
    assert summary["feat_pool_ours_vs_oracle_exact"] >= 0.995, summary
    if "grad_feat_pool" not in ref:                   # a committed record: the fp16 emulations below need the whole table
        return
    gref = ref["grad_feat_pool"]
    summary["feat_pool_oracle_exact_vs_ref"] = cosd(orc["grad_feat_pool"], gref)
    summary["feat_pool_oracle_halfprod_vs_ref"] = cosd(orc["grad_feat_pool_half_products"], gref)
    summary["feat_pool_oracle_halfaccum_vs_ref"] = cosd(orc["grad_feat_pool_half_accum"], gref)
    summary["feat_pool_tcnn_emulation_vs_exact"] = cosd(orc["grad_feat_pool_tcnn_emulation"], orc["grad_feat_pool"])
    summary["feat_pool_tcnn_emulation_vs_ref"] = cosd(orc["grad_feat_pool_tcnn_emulation"], gref)
    summary["grad_magnitudes_x128"] = orc["grad_magnitudes"]
    S = field.local_size_                                    # per level-slab agreement (fp32 element ranges [l*S, (l+2)*S))
    mine_flat, ex_flat = N(field.feat_pool_.grad).reshape(-1).astype(np.float64), np.asarray(orc["grad_feat_pool"]).reshape(-1)
    em_flat = np.asarray(orc["grad_feat_pool_tcnn_emulation"]).reshape(-1)
    slabs = []
    for l in range(17):
        sl = slice(l * S, (l + 1) * S)
        slabs.append(dict(slab=l, cos_ours_ref=cosd(mine_flat[sl], gref[sl]), cos_ours_exact=cosd(mine_flat[sl], ex_flat[sl]),
                          cos_emul_exact=cosd(em_flat[sl], ex_flat[sl]), cos_emul_ref=cosd(em_flat[sl], gref[sl]),
                          norm_ref=float(np.linalg.norm(gref[sl])), norm_ours=float(np.linalg.norm(mine_flat[sl])),
                          nnz_ref=int((gref[sl] != 0).sum()), nnz_ours=int((mine_flat[sl] != 0).sum())))
    summary["feat_pool_slabs"] = slabs
    json.dump(summary, open(diag_path("ref_grad_parity.json"), "w"), indent=1)
    for name in ("field_mlp", "shader_mlp", "app_emb"):
        assert summary[name]["cos"] >= 0.98 and summary[name]["rel_l2"] <= 0.2, (name, summary[name])
    # Ours equals the exact sum (oracle, double accumulation) to 1e-9; what is left against the reference is its own
    # fp16 noise (fp16 products + nondeterministic fp16 atomics + tcnn's fp16-accumulated dL/dinput), recorded per
    # level-slab in ref_grad_parity.json (diag_path).  (Before the RNG-stream fix in f2nerf_b200/rng.py this cosine
    # was 0.78: the TV-loss edge points were different draws.)
    assert summary["feat_pool"]["cos"] >= 0.97, summary


@pytest.mark.parametrize("ref", ["live"], indirect=True)
def test_fused_adam_vs_reference_optimizer(ref):
    """SURVEY 8f N1: f2b_adam_step against the reference's own torch::optim::Adam (C++ frontend, ExpRunner.cpp:54,136)
    stepping its own parameters with its own gradients twice — bit-identical parameters, table and MLP group."""
    if "feat_pool_after_adam" not in ref:
        pytest.skip("ref_driver without the optimizer dump")
    from f2nerf_b200._lib import call, stream
    lr = float(ref["adam_lr"][0])
    local = ((int(ref["scalars"][5]) // 16) >> 4) << 4
    table_live = 17 * local
    if "feat_pool_adam_idx" in ref:                   # a committed record: a seeded sample of the table, live entries first
        table_live = int((ref["feat_pool_adam_idx"] < table_live).sum())
    for name, wd, n_live in (("feat_pool", 0.0, table_live), ("field_mlp", 1e-6, None)):
        grad = ref["feat_pool_adam_grad"] if name == "feat_pool" and "feat_pool_adam_grad" in ref else ref["grad_" + name]
        p, g = T(ref[name + "_before_adam"]).clone(), T(grad.reshape(-1))
        m, v = torch.zeros_like(p), torch.zeros_like(p)
        n = p.numel()
        for step in (1, 2):
            call("f2b_adam_step", p, g, m, v, n, n if n_live is None else n_live, lr, 0.9, 0.99, 1e-15, wd, step, None, stream())
        want = ref[name + "_after_adam"]
        got = N(p)
        assert (got != ref[name + "_before_adam"]).any()
        np.testing.assert_array_equal(got.view(np.uint32), want.view(np.uint32), err_msg=name)


def test_ray_generation_vs_reference(ref):
    """SURVEY 8f N3: RayGenerator.RandRaysData reproduces Dataset::RandRaysData — same CPU draws under the same seed,
    bit-identical rays (Newton undistortion included), bounds and camera indices."""
    if "ds_poses" not in ref:
        pytest.skip("ref_driver without the dataset dump")
    from f2nerf_b200 import RayGenerator
    h, w = int(ref["ds_hw"][0]), int(ref["ds_hw"][1])
    gen = RayGenerator(ref["ds_poses"].reshape(-1, 3, 4), ref["ds_intri"].reshape(-1, 3, 3), ref["ds_dist_params"], ref["ds_bounds"],
                       images=None, height=h, width=w, train_set=ref["ds_train_set"].tolist())
    torch.manual_seed(2023)
    N_RAYS = n_rays_of(ref)
    (rays_o, rays_d, bounds), gt, cam = gen.RandRaysData(N_RAYS)
    assert gt is None
    bad = N(rays_d).view(np.uint32) != ref["rays_d"].view(np.uint32)
    json.dump(dict(dist_params_abs_max=float(np.abs(ref["ds_dist_params"]).max()), n_rays=int(N_RAYS),
                   frac_bad_per_component=bad.mean(0).tolist(), bad_rows=np.nonzero(bad.any(1))[0][:8].tolist(),
                   sample=[dict(row=int(r), ours=N(rays_d)[r].tolist(), ref=ref["rays_d"][r].tolist(), cam=int(ref["emb_idx"][r]),
                                ij=ref["ray_ij"][r].tolist()) for r in np.nonzero(bad.any(1))[0][:3]],
                   dist_params=ref["ds_dist_params"][:3].tolist(), intri0=ref["ds_intri"][0].tolist(), pose0=ref["ds_poses"][0].tolist()),
              open(diag_path("ref_rays.json"), "w"))
    np.testing.assert_array_equal(N(cam), ref["emb_idx"])
    np.testing.assert_array_equal(N(rays_o).view(np.uint32), ref["rays_o"].view(np.uint32))
    np.testing.assert_array_equal(N(rays_d).view(np.uint32), ref["rays_d"].view(np.uint32))
    np.testing.assert_array_equal(N(bounds), ref["ray_bounds"])
    # the kernel alone on the replayed draws
    o2, d2 = gen.Img2WorldRayFlex(T(ref["emb_idx"].astype(np.int32)), T(ref["ray_ij"]))
    np.testing.assert_array_equal(N(d2).view(np.uint32), ref["rays_d"].view(np.uint32))
    json.dump(dict(dist_params_abs_max=float(np.abs(ref["ds_dist_params"]).max()), n_rays=int(N_RAYS)),
              open(diag_path("ref_rays.json"), "w"))


def _node_fields(blob):
    """TreeNode blob -> the meaningful fields only (the reference never initialises the struct padding)."""
    t = np.ascontiguousarray(blob).view(np.uint8).reshape(-1, 64)
    return np.concatenate([t[:, :53], t[:, 56:60]], 1)


def test_octree_maintenance_vs_reference(ref, oracle):
    """SURVEY 8f N2: the device ProcOctree / MarkInvisibleNodes against the reference's own host pass on its ngp_fox octree
    (every 5th valid leaf killed, synthetic visit counts): subdivide -> mark invisible -> compact, byte-identical blobs."""
    if "oct_nodes_in" not in ref:
        pytest.skip("ref_driver without the octree dump")
    gdp, sampler, field, shader, renderer = build_from_ref(ref)
    sampler.tree_nodes_gpu_, sampler.tree_weight_stats_ = T(ref["oct_nodes_in"]), T(ref["oct_w_in"])
    sampler.tree_alpha_stats_, sampler.tree_visit_cnt_ = T(ref["oct_a_in"]), T(ref["oct_visit_in"])
    on, ow, oa = oracle.octree_proc(ref["oct_nodes_in"], ref["oct_w_in"], ref["oct_a_in"], ref["oct_visit_in"], True, False)
    np.testing.assert_array_equal(_node_fields(on), _node_fields(ref["oct_nodes_sub"]))    # the sequential restatement first
    m = sampler.ProcOctree(True, True, False)
    assert m == ref["oct_nodes_sub"].size // 64
    np.testing.assert_array_equal(_node_fields(N(sampler.tree_nodes_gpu_)), _node_fields(ref["oct_nodes_sub"]))
    np.testing.assert_array_equal(N(sampler.tree_weight_stats_), ref["oct_w_sub"])
    np.testing.assert_array_equal(N(sampler.tree_alpha_stats_), ref["oct_a_sub"])
    sampler.MarkInvisibleNodes(ref["oct_intri"].reshape(-1, 3, 3), ref["oct_w2c"].reshape(-1, 3, 4), ref["oct_bound"])
    mine = N(sampler.tree_nodes_gpu_).view(np.int32).reshape(-1, 16)[:, 14]
    theirs = ref["oct_nodes_invis"].view(np.int32).reshape(-1, 16)[:, 14]
    flips = int(((mine < 0) != (theirs < 0)).sum())
    json.dump(dict(nodes=int(m), invisible_ref=int((theirs < 0).sum()), invisible_ours=int((mine < 0).sum()), flips=flips),
              open(diag_path("ref_octree.json"), "w"))
    assert flips <= max(1, m // 2000), flips                                     # fp32 visibility tests: borderline nodes only
    sampler.tree_nodes_gpu_ = T(ref["oct_nodes_invis"])                          # continue from the reference's own marks
    m = sampler.ProcOctree(True, False, False)
    np.testing.assert_array_equal(_node_fields(N(sampler.tree_nodes_gpu_)), _node_fields(ref["oct_nodes_final"]))
    np.testing.assert_array_equal(N(sampler.tree_weight_stats_), ref["oct_w_final"])
    np.testing.assert_array_equal(N(sampler.tree_alpha_stats_), ref["oct_a_final"])


def test_sh_encode_bit_exact_vs_reference(ref):
    """f2b_sh_encode (and with it the fused shader-input epilogue, which shares the device function) == SHKenerl bit for bit."""
    from f2nerf_b200 import ops
    got = ops.sh_encode(T(ref["val_dirs"]))
    np.testing.assert_array_equal(N(got).view(np.uint32), ref["val_sh"].view(np.uint32))


def test_mark_invisible_vs_reference(ref, oracle):
    """f2b_octree_mark_invisible == the reference's MarkInvisibleNodes on its subdivided octree == the oracle restatement."""
    gdp, sampler, field, shader, renderer = build_from_ref(ref)
    sampler.tree_nodes_gpu_ = T(np.ascontiguousarray(ref["oct_nodes_sub"]).view(np.uint8).reshape(-1))
    sampler.MarkInvisibleNodes(ref["oct_intri"].reshape(-1, 3, 3), ref["oct_w2c"].reshape(-1, 3, 4), ref["oct_bound"])
    mine = N(sampler.tree_nodes_gpu_).view(np.int32).reshape(-1, 16)[:, 14]
    theirs = np.ascontiguousarray(ref["oct_nodes_invis"]).view(np.uint8).view(np.int32).reshape(-1, 16)[:, 14]
    orc = oracle.mark_invisible(ref["oct_nodes_sub"], ref["oct_intri"], ref["oct_w2c"], ref["oct_bound"]).view(np.int32).reshape(-1, 16)[:, 14]
    np.testing.assert_array_equal(mine, orc)
    np.testing.assert_array_equal(mine, theirs)
