"""f2b_field_bwd_scatter (field-MLP backward + hash-table scatter in one kernel) against the two-kernel sequence it replaces
(f2b_mlp_bwd2 -> fp16 dL/dfeatures in memory -> f2b_hash_bwd per point segment) and against the CPU oracle's exact scatter.

The fused kernel rounds dL/dfeatures to the same fp16 bits and forms the same per-run sums, so the two paths differ only in the
order of their fp32 reductions: relative L2 <= 1e-6 on both gradients.  (The weight gradient is accumulated in TMEM over chains of
tiles; the fused kernel flushes after as many tiles as a CTA of f2b_mlp_bwd2 accumulates, so its rounding matches.)"""
import numpy as np
import pytest
import torch

from conftest import make_rays
from test_gpu_parity import N, T, assert_close

pytestmark = pytest.mark.gpu

DEV = "cuda"


def rel_l2(a, b):
    a, b = a.double(), b.double()
    return float(torch.linalg.norm(a - b) / max(float(torch.linalg.norm(b)), 1e-300))


def ray_points(n, V, seed):
    """n points in [-1, 1]^3 laid out like a ray batch: runs of consecutive samples a short step apart (the coarse levels merge
    runs of lanes), one volume per ray."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    ray = torch.arange(n, device=DEV) // 97
    n_rays = int(ray[-1]) + 1 if n else 0
    start = torch.rand((n_rays, 3), device=DEV, generator=g) * 1.6 - .8
    step = (torch.rand((n_rays, 3), device=DEV, generator=g) - .5) * 4e-3
    k = (torch.arange(n, device=DEV) % 97).float()[:, None]
    pts = (start[ray] + k * step[ray]).contiguous()
    vol = torch.randint(0, V, (n_rays,), device=DEV, generator=g, dtype=torch.int32)[ray]
    return pts, vol


def make_inputs(n_kept, n_edge, hp, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    n = n_kept + n_edge
    # positive-biased dL/dout: the weight-gradient sums do not cancel, so their relative error measures summation order only
    dout = (torch.randn((n, 16), device=DEV, generator=g) * .1 + .05).half()
    dout[5::11] = 0                                                    # zero-gradient rows are skipped by the scatter
    x = (torch.randn((n, 32), device=DEV, generator=g) * .5).half()
    pts, vol = ray_points(n_kept, hp["V"], seed + 1)
    anchors = torch.stack([vol, torch.zeros_like(vol), torch.zeros_like(vol)], 1).contiguous()   # volume in column 0 of 3
    e_pts, e_anc = ray_points(n_edge, hp["V"], seed + 2)
    return dout.contiguous(), x.contiguous(), pts, anchors, e_pts, e_anc


def two_kernel(dout, x, params, pts, anchors, e_pts, e_anc, hp, grad_mul):
    from f2nerf_b200 import ops
    from f2nerf_b200._lib import call, stream
    n_kept, n = pts.shape[0], dout.shape[0]
    din = torch.empty((n, 32), dtype=torch.float16, device=DEV)
    dp = torch.zeros(params.numel(), dtype=torch.float32, device=DEV)
    table = torch.zeros((hp["pool"], 2), dtype=torch.float32, device=DEV)
    args = (T(hp["prim"]), T(hp["bias"]), hp["V"], hp["local_size"])
    for s0, s1, p, a, stride in ((0, n_kept, pts, anchors, 3), (n_kept, n, e_pts, e_anc, 1)):
        if s1 > s0:
            call("f2b_mlp_bwd2", dout[s0:s1], x[s0:s1], None, None, params, 0, s1 - s0, din[s0:s1], dp, stream())
            ops.hash_bwd(*args, p, a, stride, din[s0:s1], grad_mul, table)
    return din, dp, table


def fused(dout, x, params, pts, anchors, e_pts, e_anc, hp, grad_mul):
    from f2nerf_b200 import ops
    dp = torch.zeros(params.numel(), dtype=torch.float32, device=DEV)
    table = torch.zeros((hp["pool"], 2), dtype=torch.float32, device=DEV)
    ops.field_bwd_scatter(dout, x, params, pts, anchors, e_pts if e_pts.shape[0] else None, e_anc if e_anc.shape[0] else None,
                          T(hp["prim"]), T(hp["bias"]), hp["V"], hp["local_size"], grad_mul, dp, table)
    return dp, table


@pytest.mark.parametrize("n_kept,n_edge", [(1, 0), (127, 0), (128, 0), (129, 0), (0, 200), (1013, 300), (4096 + 77, 16384),
                                           (3_100_000, 16384)])
def test_matches_two_kernel_sequence(oracle, hash_params, n_kept, n_edge):
    hp = hash_params
    params = T((oracle.mlp_init(32, 0) * 2).astype(np.float16))
    dout, x, pts, anchors, e_pts, e_anc = make_inputs(n_kept, n_edge, hp, seed=n_kept + 7 * n_edge)
    _, dp_a, table_a = two_kernel(dout, x, params, pts, anchors, e_pts, e_anc, hp, 0.5)
    dp_b, table_b = fused(dout, x, params, pts, anchors, e_pts, e_anc, hp, 0.5)
    assert float(table_a.abs().max()) > 0
    assert rel_l2(dp_b, dp_a) <= 1e-6, rel_l2(dp_b, dp_a)
    assert rel_l2(table_b, table_a) <= 1e-6, rel_l2(table_b, table_a)
    # only the first 17/32 of the pool is ever touched (half-overlapping levels)
    assert float(table_b[(17 * hp["local_size"]) // 2 + 1:].abs().max()) == 0.0


def test_table_gradient_matches_oracle(scene, oracle, hash_params):
    """The scatter of the kernel's own fp16 dL/dfeatures (the same bits f2b_mlp_bwd2 returns) against the oracle's exact sum,
    ray samples from the oracle's sampler plus an edge segment that starts off a 32-row boundary."""
    from f2nerf_b200 import ops
    hp = hash_params
    o, d, dn, _ = make_rays(scene, 32, seed=11)
    s = oracle.sampler(scene["nodes"], scene["trans"], o, dn, np.ones(1024 + 32 + 10, np.float32), 0.05, 1e8, 1 / 256, False, 1024)
    n_kept = s["pts"].shape[0]
    n_edge = 333
    params = T((oracle.mlp_init(32, 0) * 2).astype(np.float16))
    dout, x, _, _, e_pts, e_anc = make_inputs(n_kept, n_edge, hp, seed=5)
    pts, anchors = T(s["pts"]), T(s["anchors"])
    din, _, _ = two_kernel(dout, x, params, pts, anchors, e_pts, e_anc, hp, 0.5)
    _, table = fused(dout, x, params, pts, anchors, e_pts, e_anc, hp, 0.5)
    scales = ops.hash_level_scales().numpy()
    g = N(din).astype(np.float32)
    ref = oracle.hash_bwd(hp["prim"], hp["bias"], hp["V"], hp["local_size"], scales, s["pts"], s["anchors"], 3, g[:n_kept], 0.5,
                          hp["pool"])
    ref += oracle.hash_bwd(hp["prim"], hp["bias"], hp["V"], hp["local_size"], scales, N(e_pts), N(e_anc), 1, g[n_kept:], 0.5,
                           hp["pool"])
    assert_close(N(table), ref, rtol=1e-4, atol_frac=1e-5, name="field_bwd_scatter table gradient")


def test_nonfinite_row_reaches_flag(oracle, hash_params):
    """A NaN dL/dout row stays live in the scatter: the table gradient turns non-finite and f2b_render_grad_finalize raises the
    field MLP's flag."""
    from f2nerf_b200 import _lib
    from f2nerf_b200._lib import call
    hp = hash_params
    params = T((oracle.mlp_init(32, 0) * 2).astype(np.float16))
    dout, x, pts, anchors, e_pts, e_anc = make_inputs(1000, 64, hp, seed=3)
    dout[517] = float("nan")
    dp, table = fused(dout, x, params, pts, anchors, e_pts, e_anc, hp, 0.5)
    assert not bool(torch.isfinite(table).all())
    d_sparams = torch.zeros(16, dtype=torch.float32, device=DEV)
    flags = torch.zeros(2, dtype=torch.int32, device=DEV)
    dp_finite = torch.zeros_like(dp)                                  # only the table gradient can raise the flag here
    ra = _lib.RenderArgs().set(d_sparams=d_sparams, n_shader_params=16, d_fparams=dp_finite, n_field_params=dp.numel(),
                               d_table=table, table_live=table.numel(), nonfinite=flags, shader_loss_scale=1., field_loss_scale=1.,
                               app_emb=None, ray_emb_idx=None, stream=torch.cuda.current_stream().cuda_stream)
    call("f2b_render_grad_finalize", ra)
    assert N(flags).tolist() == [0, 1]
