#!/usr/bin/env python
"""Generate the committed golden fixtures under tests/golden/ by running the UNMODIFIED reference
(oracle/_ref/ref_driver, built by oracle/Makefile.ref) and the same program with the B200 drop-in linked in
(oracle/_ref/ref_driver_b200) on a B200:

    python oracle/make_golden.py [OUT_DIR]            # default OUT_DIR: tests/golden

ref_ngp_fox.npz holds the reference's own ngp_fox octree / warp blobs, a small seeded ray batch and every
boundary tensor of PersSampler::GetSamples, Hash3DAnchored::AnchoredQuery, SHShader::Query and
Renderer::Render for it (VALIDATE mode, plus the seeded TRAIN-mode sampler outputs and octree statistics).
tests/test_golden_ref.py pins oracle/f2_oracle.c against it on the CPU.  The 64 MB hash table is not stored:
both sides regenerate it from the CPU generator seed 1234 (see ref_driver.cpp).

ref_ngp_fox_512.npz (the reference) and shim_fused_512.npz (the fused C++ host inside the reference's program) record
the 512-ray run that tests/test_ref_parity.py ("live") and tests/test_shim_dropin.py compare against where the binaries
are not built.  Each stays under 1 MB: per-ray outputs are whole, per-sample outputs and the table gradient are seeded
samples (the kept rows are stored beside them as ``*_idx``), and what equals ref_ngp_fox.npz (warps, parameters,
cameras, octree-maintenance dumps) is stored once, there, and named in ``from_ref_ngp_fox``.
"""
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N_RAYS = 40
N_RAYS_RECORD = 512
MAX_BYTES = 1_000_000


def run_driver(binary, n_rays, out, env=None):
    """The driver's dumps of one seeded run (``<n_rays> 0 1``: no timing, full table gradient), keyed by file name."""
    r = subprocess.run([os.path.join(ROOT, "oracle", "_ref", binary), os.path.join(ROOT, "oracle", "ref_config_ngp_fox.yaml"), out,
                        str(n_rays), "0", "1"], cwd=ROOT, capture_output=True, text=True, timeout=900, env=env)
    if r.returncode != 0:
        print(r.stdout[-2000:], r.stderr[-4000:])
        sys.exit(1)
    return {f[:-4]: np.load(os.path.join(out, f)) for f in os.listdir(out) if f.endswith(".npy")}


def table_grad_sample(g, scalars, n, seed):
    """The hash-table gradient (64 MB dense) as a seeded n-element subsample of its live prefix + per-level-slab norms."""
    g = g.reshape(-1)
    local = ((int(scalars[5]) // 16) >> 4) << 4
    assert not g[17 * local:].any()
    sub = np.sort(np.random.default_rng(seed).choice(17 * local, n, replace=False)).astype(np.int64)
    return {"grad_feat_pool_sub_idx": sub, "grad_feat_pool_sub_val": g[sub].astype(np.float32),
            "grad_feat_pool_slab_norm": np.array([np.linalg.norm(g[l * local:(l + 1) * local].astype(np.float64)) for l in range(17)],
                                                 np.float32)}


def fixture(out_dir):
    d = run_driver("ref_driver", N_RAYS, "/tmp/f2b_golden_dump")
    keep = ["tree_nodes", "pers_trans", "edge_pool", "search_order", "prim_pool", "bias_pool", "field_mlp_params",
            "shader_mlp_params", "app_emb", "scalars", "rays_o", "rays_d", "rays_d_normed", "gt_colors", "emb_idx",
            "val_pts", "val_dirs", "val_dt", "val_t", "val_anchors", "val_bounds", "val_first_oct_dis", "val_scene_feat",
            "val_rgb", "val_sh", "val_colors", "val_disparity", "val_depth", "val_weights", "val_idx_start_end",
            "train_noise", "train_bg", "train_edge_idx", "train_edge_coord", "train_pts", "train_dt", "train_t", "train_anchors",
            "train_bounds", "train_colors", "train_disparity", "train_depth", "train_weights", "train_idx_start_end",
            "train_first_oct_dis", "train_tree_nodes_after", "train_weight_stats_after", "train_alpha_stats_after",
            "train_visit_cnt_after", "train_loss", "grad_field_mlp", "grad_shader_mlp", "grad_app_emb",
            "edge_idx", "edge_coord", "edge_pts", "edge_anchors", "train_edge_feats",
            "ds_poses", "ds_intri", "ds_dist_params", "ray_ij", "ds_hw", "ds_bounds", "ds_train_set", "ray_bounds",
            "oct_intri", "oct_w2c", "oct_bound", "backward_nan",
            "oct_nodes_in", "oct_w_in", "oct_a_in", "oct_visit_in", "oct_nodes_sub", "oct_w_sub", "oct_a_sub",
            "oct_nodes_invis", "oct_nodes_final", "oct_w_final", "oct_a_final"]
    data = {k: d[k] for k in keep}
    for k in ("edge_idx", "edge_coord", "edge_pts", "edge_anchors"):         # 2048 of the 8192 draws are plenty
        data[k] = np.ascontiguousarray(data[k][:2048])
    data.update(table_grad_sample(d["grad_feat_pool"], data["scalars"], 1 << 18, 0))
    data["train_edge_feats"] = np.ascontiguousarray(data["train_edge_feats"][:2048]).astype(np.float16)   # fp16 values
    # the level scales as the device computes them (MUFU.EX2): the oracle takes them as an input
    sys.path.insert(0, ROOT)
    from f2nerf_b200 import ops
    data["level_scales"] = ops.hash_level_scales().numpy()
    data["val_scene_feat"] = data["val_scene_feat"].astype(np.float16)       # tcnn outputs are fp16 values
    data["train_edge_coord"] = data["train_edge_coord"].astype(np.float32)
    save(os.path.join(out_dir, "ref_ngp_fox.npz"), data, limit=None)


def rows(data, idx_key, keys, n, seed):
    """Keep a seeded sample of n rows (sorted) of the per-sample arrays ``keys`` (same row count); the rows go to ``idx_key``."""
    total = data[keys[0]].shape[0]
    idx = np.sort(np.random.default_rng(seed).choice(total, min(n, total), replace=False)).astype(np.int32)
    for k in keys:
        assert data[k].shape[0] == total, k
        data[k] = np.ascontiguousarray(data[k][idx])
    data[idx_key] = idx


def node_fields(blob):
    """TreeNode blob -> the meaningful fields only (the reference never initialises the struct padding)."""
    t = np.ascontiguousarray(blob).view(np.uint8).reshape(-1, 64)
    return np.concatenate([t[:, :53], t[:, 56:60]], 1)


def shared_with_fixture(data, gold):
    """Move the entries the 40-ray fixture holds too (warps, parameters, cameras, octree-maintenance dumps) out of ``data``.
    The octree-maintenance blobs count as equal when their fields are (the tests that read them compare fields only); the
    march's own octree stays whatever its padding bytes: they reach train_tree_nodes_after, which is compared byte for byte."""
    def same(k):
        a, b = gold[k], data[k]
        if a.shape != b.shape or a.dtype != b.dtype:
            return False
        return np.array_equal(node_fields(a), node_fields(b)) if k.startswith("oct_nodes") else np.array_equal(a, b)
    shared = [k for k in gold if k in data and same(k)]
    for k in ("prim_pool", "bias_pool", "field_mlp_params", "shader_mlp_params", "app_emb"):
        assert k in shared, f"{k}: the {N_RAYS_RECORD}-ray run does not share the fixture's parameters"
    for k in shared:
        del data[k]
    data["from_ref_ngp_fox"] = np.array(sorted(shared))


def record_ref(d, gold):
    """The reference's 512-ray run for tests/test_ref_parity.py."""
    data = {k: v for k, v in d.items() if not k.startswith(("grad_feat_pool", "feat_pool_", "ray_cam_draw"))}
    rows(data, "val_sample_idx", ["val_pts", "val_dirs", "val_dt", "val_t", "val_anchors", "val_scene_feat", "val_rgb", "val_sh"], 512, 1)
    rows(data, "train_sample_idx", ["train_pts", "train_dt", "train_t", "train_anchors"], 512, 2)
    rows(data, "val_weights_idx", ["val_weights"], 512, 3)
    del data["train_weights"]                                                # no test reads it
    data["val_scene_feat"] = data["val_scene_feat"].astype(np.float16)       # tcnn outputs are fp16 values
    for k in ("edge_idx", "edge_coord", "edge_pts", "edge_anchors"):
        data[k] = np.ascontiguousarray(data[k][:2048])
    data["train_edge_feats"] = np.ascontiguousarray(data["train_edge_feats"][:512]).astype(np.float16)
    data.update(table_grad_sample(d["grad_feat_pool"], d["scalars"], 1 << 12, 0))
    # torch::optim::Adam is elementwise: its two steps on a seeded sample of the table (live prefix first, then dead entries,
    # which it must leave alone) pin the fused optimizer as well as the whole table does
    local = ((int(d["scalars"][5]) // 16) >> 4) << 4
    n_all = d["feat_pool_before_adam"].size
    rng = np.random.default_rng(5)
    live = np.sort(rng.choice(17 * local, 1024, replace=False))
    dead = np.sort(rng.choice(np.arange(17 * local, n_all), 256, replace=False))
    idx = np.concatenate([live, dead]).astype(np.int64)
    data["feat_pool_adam_idx"] = idx
    for k in ("feat_pool_before_adam", "feat_pool_after_adam"):
        data[k] = d[k].reshape(-1)[idx]
    data["feat_pool_adam_grad"] = d["grad_feat_pool"].reshape(-1)[idx]
    data["field_mlp_before_adam"], data["field_mlp_after_adam"] = d["field_mlp_before_adam"], d["field_mlp_after_adam"]
    shared_with_fixture(data, gold)
    return data


def record_fused(d, gold):
    """ref_driver_b200's 512-ray TRAIN step (the fused C++ host) for tests/test_shim_dropin.py: its inputs and every output the
    Python host is compared with."""
    keep = ["scalars", "rays_o", "rays_d", "emb_idx", "gt_colors", "tree_nodes", "pers_trans", "edge_pool", "prim_pool", "bias_pool",
            "field_mlp_params", "shader_mlp_params", "app_emb", "train_idx_start_end", "train_colors", "train_disparity", "train_depth",
            "train_weights", "train_edge_feats", "train_first_oct_dis", "train_weight_stats_after", "train_alpha_stats_after",
            "train_visit_cnt_after", "train_tree_nodes_after", "train_loss", "grad_field_mlp", "grad_shader_mlp", "grad_app_emb"]
    data = {k: d[k] for k in keep}
    rows(data, "train_weights_idx", ["train_weights"], 1024, 4)
    rows(data, "train_edge_feats_idx", ["train_edge_feats"], 256, 6)
    data.update(table_grad_sample(d["grad_feat_pool"], d["scalars"], 1 << 12, 0))
    shared_with_fixture(data, gold)
    return data


def records(out_dir):
    gold = dict(np.load(os.path.join(ROOT, "tests", "golden", "ref_ngp_fox.npz")))
    d = run_driver("ref_driver", N_RAYS_RECORD, "/tmp/f2b_record_ref")
    save(os.path.join(out_dir, "ref_ngp_fox_512.npz"), record_ref(d, gold))
    env = {k: v for k, v in os.environ.items() if k not in ("F2B_SHIM", "F2B_RENDER")}
    d = run_driver("ref_driver_b200", N_RAYS_RECORD, "/tmp/f2b_record_fused", env)
    save(os.path.join(out_dir, "shim_fused_512.npz"), record_fused(d, gold))


def save(dst, data, limit=MAX_BYTES):
    os.makedirs(os.path.dirname(dst), exist_ok=True)
    np.savez_compressed(dst, **data)
    size = os.path.getsize(dst)
    print("wrote", dst, size / 1e6, "MB")
    assert limit is None or size <= limit, f"{dst}: {size} bytes, over the {limit}-byte budget of a committed fixture"


def main():
    out_dir = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden")
    fixture(out_dir)
    records(out_dir)


if __name__ == "__main__":
    main()
