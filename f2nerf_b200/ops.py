"""Thin allocation wrappers over the C ABI (one python function per entry point) plus the reference's
free-function operator surface: ``FlexOps.Sum / AccumulateSum`` (``FlexOps.h:15-16``),
``CustomOps.WeightVar / GradientScaling / ScatterAdd / ScatterIdx`` (``CustomOps.h:24-25``,
``Scatter.h:16-17``) and ``TruncExp`` (``CustomOps.h:12-18``), with the same argument meaning.

Everything here runs on CUDA through libf2nerf_b200.so; there is no CPU path.
"""
import torch

from . import _lib
from ._lib import call, stream

F16, F32, I32, U8 = torch.float16, torch.float32, torch.int32, torch.uint8


def _chk(t, dtype, name):
    if not t.is_cuda:
        raise ValueError(f"{name}: expected a CUDA tensor (the reference's CHECK_TS / CUDA* options)")
    if t.dtype != dtype:
        raise ValueError(f"{name}: expected dtype {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError(f"{name}: expected a contiguous tensor (the reference's CK_CONT)")
    return t


def dev_empty(shape, dtype, like):
    return torch.empty(shape, dtype=dtype, device=like.device)


# ------------------------------------------------------------------ sampler ---------------------
def sampler_count(tree_nodes, trans, rays_o, rays_d, noise, near, far, sample_l, scale_by_dis, max_hits, count_all_hits=True):
    R = rays_o.shape[0]
    counts = dev_empty((max(R, 1),), I32, rays_o)
    bounds = dev_empty((R, 2), I32, rays_o)
    totals = dev_empty((2,), I32, rays_o)
    call("f2b_sampler_count", tree_nodes, tree_nodes.numel() // 64, trans, trans.numel() // 544, rays_o, rays_d,
         noise, R, float(near), float(far), float(sample_l), int(bool(scale_by_dis)), int(max_hits), int(bool(count_all_hits)),
         counts, bounds, totals, stream())
    return bounds, totals


def sampler_fill(tree_nodes, trans, rays_o, rays_d, noise, near, far, sample_l, scale_by_dis, max_hits, bounds, n_pts):
    R = rays_o.shape[0]
    pts = dev_empty((n_pts, 3), F32, rays_o)
    dirs = dev_empty((n_pts, 3), F32, rays_o)
    dt = dev_empty((n_pts,), F32, rays_o)
    t = dev_empty((n_pts,), F32, rays_o)
    anchors = dev_empty((n_pts, 3), I32, rays_o)
    first = dev_empty((R, 1), F32, rays_o)
    call("f2b_sampler_fill", tree_nodes, tree_nodes.numel() // 64, trans, trans.numel() // 544, rays_o, rays_d, noise,
         R, float(near), float(far), float(sample_l), int(bool(scale_by_dis)), int(max_hits), bounds, pts, dirs, dt, t,
         anchors, first, stream())
    return pts, dirs, dt, t, anchors, first


def sampler_march(tree_nodes, trans, rays_o, rays_d, noise, near, far, sample_l, scale_by_dis, max_hits, scratch,
                  count_all_hits=False):
    """One-pass march into per-ray scratch slots -> (bounds, totals, first_oct_dis).  scratch = (s_pts, s_dt, s_t, s_anchors)."""
    R = rays_o.shape[0]
    counts = dev_empty((max(R, 1),), I32, rays_o)
    bounds = dev_empty((R, 2), I32, rays_o)
    totals = dev_empty((2,), I32, rays_o)
    first = dev_empty((R, 1), F32, rays_o)
    call("f2b_sampler_march", tree_nodes, tree_nodes.numel() // 64, trans, trans.numel() // 544, rays_o, rays_d, noise, R,
         float(near), float(far), float(sample_l), int(bool(scale_by_dis)), int(max_hits), int(bool(count_all_hits)),
         *scratch, counts, bounds, totals, first, stream())
    return bounds, totals, first


def sampler_gather(rays_d, bounds, n_pts, scratch):
    pts = dev_empty((n_pts, 3), F32, rays_d)
    dirs = dev_empty((n_pts, 3), F32, rays_d)
    dt = dev_empty((n_pts,), F32, rays_d)
    t = dev_empty((n_pts,), F32, rays_d)
    anchors = dev_empty((n_pts, 3), I32, rays_d)
    call("f2b_sampler_gather", rays_d, bounds, bounds.shape[0], *scratch, pts, dirs, dt, t, anchors, stream())
    return pts, dirs, dt, t, anchors


def edge_samples(edge_pool, trans, edge_idx, edge_coord):
    n = edge_idx.shape[0]
    out_pts = dev_empty((n, 2, 3), F32, edge_coord)
    out_idx = dev_empty((n, 2), I32, edge_coord)
    call("f2b_edge_samples", edge_pool, trans, edge_idx, edge_coord, n, out_pts, out_idx, stream())
    return out_pts, out_idx


# ------------------------------------------------------------------ field -----------------------
def hash_level_scales():
    import ctypes
    buf = (ctypes.c_float * 16)()
    call("f2b_hash_level_scales", ctypes.addressof(buf))
    return torch.tensor(list(buf), dtype=F32)


def table_to_half(table_f32):
    out = torch.empty_like(table_f32, dtype=F16)
    call("f2b_table_to_half", table_f32, out, table_f32.numel(), stream())
    return out


def hash_fwd(table_f16, prim_pool, bias_pool, n_volumes, local_size, pts, vol, vol_stride=1):
    n = pts.shape[0]
    out = dev_empty((n, 32), F16, pts)
    call("f2b_hash_fwd", table_f16, prim_pool, bias_pool, int(n_volumes), int(local_size), pts, vol, int(vol_stride), n,
         out, stream())
    return out


def hash_bwd(prim_pool, bias_pool, n_volumes, local_size, pts, vol, vol_stride, grad_feat, grad_mul, grad_table):
    n = pts.shape[0]
    call("f2b_hash_bwd", prim_pool, bias_pool, int(n_volumes), int(local_size), pts, vol, int(vol_stride), n,
         grad_feat, int(grad_feat.dtype == F16), float(grad_mul), grad_table, stream())
    return grad_table


def field_bwd_scatter(d_out16, feat16, params16, pts, anchors, e_pts, e_anc, prim_pool, bias_pool, n_volumes, local_size, grad_mul,
                      d_params, grad_table):
    """Field-MLP backward (0 hidden matmuls) + hash scatter in one kernel.  Rows [0, len(pts)) of d_out16 [P,16] / feat16 [P,32]
    are samples at pts [.,3] / anchors [.,3] (volume = column 0), the rest edge points at e_pts / e_anc [.] (None when there are
    none).  d_params and grad_table are accumulated into."""
    n_kept, n_edge = pts.shape[0], d_out16.shape[0] - pts.shape[0]
    if n_edge and (e_pts is None or e_pts.shape[0] != n_edge):
        raise ValueError("field_bwd_scatter: edge rows without their edge points")
    call("f2b_field_bwd_scatter", d_out16, feat16, params16, n_kept, pts, anchors, n_edge, e_pts, e_anc, prim_pool, bias_pool,
         int(n_volumes), int(local_size), float(grad_mul), d_params, grad_table, stream())
    return d_params, grad_table


def field_fwd(table_f16, prim_pool, bias_pool, n_volumes, local_size, params_f16, pts, vol, vol_stride=1, logit_only=False,
              save=False, save_feat=None):
    """Fused hash encode + tcgen05 field MLP.  -> (out [n] or [n,16] fp32, feat16 | None, hidden | None).
    ``save`` keeps features + hidden activations (gradient pass); ``save_feat`` keeps only the features."""
    n = pts.shape[0]
    save_feat = save if save_feat is None else save_feat
    out = dev_empty((n,) if logit_only else (n, 16), F32, pts)
    feat = dev_empty((n, 32), F16, pts) if save_feat else None
    hidden = dev_empty((1, n, 64), F16, pts) if (save and not logit_only) else None
    call("f2b_field_fwd", table_f16, prim_pool, bias_pool, int(n_volumes), int(local_size), params_f16, pts, vol,
         int(vol_stride), n, int(bool(logit_only)), out, feat, hidden, stream())
    return out, feat, hidden


def mlp_fwd(x_f16, params_f16, n_hidden_matmuls, save_hidden=False, impl=None):
    n = x_f16.shape[0]
    out = dev_empty((n, 16), F16, x_f16)
    hidden = dev_empty((n_hidden_matmuls + 1, n, 64), F16, x_f16) if save_hidden else None
    name = "f2b_mlp_fwd" if impl is None else f"f2b_mlp_fwd_{impl}"
    call(name, x_f16, params_f16, int(n_hidden_matmuls), n, out, hidden, stream())
    return out, hidden


def mlp_fwd_f32(x_f16, params_f16, n_hidden_matmuls, save_hidden=False, want_f16=False):
    """MLP forward returning fp32 [n,16] (fp16-rounded values) straight from the epilogue: -> (out32, out16|None, hidden)."""
    from . import _lib
    n = x_f16.shape[0]
    out32 = dev_empty((n, 16), F32, x_f16)
    out16 = dev_empty((n, 16), F16, x_f16) if (want_f16 or _lib.lib.f2b_get_mlp_impl() != 1) else None
    hidden = dev_empty((n_hidden_matmuls + 1, n, 64), F16, x_f16) if save_hidden else None
    call("f2b_mlp_fwd_f32", x_f16, params_f16, int(n_hidden_matmuls), n, out32, out16, hidden, stream())
    return out32, out16, hidden


def mlp_bwd(dout_f16, x_f16, hidden, params_f16, n_hidden_matmuls, need_din=True, impl=None):
    n = x_f16.shape[0]
    din = dev_empty((n, 32), F16, x_f16) if need_din else None
    dparams = torch.zeros(params_f16.numel(), dtype=F32, device=x_f16.device)
    name = "f2b_mlp_bwd" if impl is None else f"f2b_mlp_bwd_{impl}"
    call(name, dout_f16, x_f16, hidden, params_f16, int(n_hidden_matmuls), n, din, dparams, stream())
    return din, dparams


def cast_f32_to_f16(x, scale=1.0):
    out = torch.empty_like(x, dtype=F16)
    call("f2b_cast_f32_to_f16", x, out, x.numel(), float(scale), stream())
    return out


def cast_f16_to_f32(x, scale=1.0):
    out = torch.empty_like(x, dtype=F32)
    call("f2b_cast_f16_to_f32", x, out, x.numel(), float(scale), stream())
    return out


# ------------------------------------------------------------------ shader ----------------------
def sh_encode(dirs, degree=4):
    n = dirs.shape[0]
    out = dev_empty((n, degree * degree), F32, dirs)
    call("f2b_sh_encode", dirs, n, int(degree), out, stream())
    return out


def scatter_idx(n_all_pts, idx_start_end, emb_idx):
    out = dev_empty((n_all_pts,), I32, idx_start_end)
    call("f2b_scatter_idx", idx_start_end, emb_idx, idx_start_end.shape[0], out, stream())
    return out


def shader_prep(scene_feat, dirs, app_emb=None, pt_emb_idx=None):
    n = scene_feat.shape[0]
    out = dev_empty((n, 32), F16, scene_feat)
    call("f2b_shader_prep", scene_feat, dirs, app_emb, pt_emb_idx, n, out, stream())
    return out


def shader_act(raw_f16):
    n = raw_f16.shape[0]
    rgb = dev_empty((n, 3), F32, raw_f16)
    call("f2b_shader_act", raw_f16, n, rgb, stream())
    return rgb


def shader_act_bwd(raw_f16, d_rgb, loss_scale):
    n = raw_f16.shape[0]
    out = dev_empty((n, 16), F16, raw_f16)
    call("f2b_shader_act_bwd", raw_f16, d_rgb, n, float(loss_scale), out, stream())
    return out


def shader_prep_bwd(d_mlp_in_f16, bounds, emb_idx, inv_loss_scale, d_scene_feat, d_app_emb):
    call("f2b_shader_prep_bwd", d_mlp_in_f16, bounds, emb_idx, bounds.shape[0], float(inv_loss_scale), d_scene_feat,
         d_app_emb, stream())


def shader_prep_bwd_f16(d_mlp_in_f16, d_logit, bounds, emb_idx, inv_loss_scale, field_loss_scale, d_field_out_f16, d_app_emb):
    """Fused tail of the shader backward: writes the field MLP's dL/dout (fp16, loss-scaled) for the first
    len(d_logit) rows of ``d_field_out_f16`` and accumulates d_app_emb."""
    call("f2b_shader_prep_bwd_f16", d_mlp_in_f16, d_logit, bounds, emb_idx, bounds.shape[0], float(inv_loss_scale),
         float(field_loss_scale), d_field_out_f16, d_app_emb, stream())


# ------------------------------------------------------------------ composite -------------------
def early_stop(logit, logit_stride, dt, bounds):
    R, P = bounds.shape[0], dt.shape[0]
    weights, alphas = dev_empty((P,), F32, dt), dev_empty((P,), F32, dt)
    keep = dev_empty((P,), U8, dt)
    counts = dev_empty((max(R, 1),), I32, dt)
    new_bounds = dev_empty((R, 2), I32, dt)
    total = dev_empty((1,), I32, dt)
    call("f2b_early_stop", logit, int(logit_stride), dt, bounds, R, weights, alphas, keep, counts, new_bounds, total,
         stream())
    return weights, alphas, keep, new_bounds, total


def field_fwd_slots(table_f16, prim_pool, bias_pool, n_volumes, local_size, params_f16, slot_pts, slot_anchors, counts, n_rays,
                    slot, out_logit, feat_slots):
    """Early-stop field pass over the march's slot layout (logit only); all tensor arguments may be ray-chunk views."""
    call("f2b_field_fwd_slots", table_f16, prim_pool, bias_pool, int(n_volumes), int(local_size), params_f16, slot_pts,
         slot_anchors, int(slot_anchors.shape[1]), counts, int(n_rays), int(slot), 1, out_logit, feat_slots, stream())


def early_stop_rays(logit, logit_stride, dt, bounds, weights, alphas, keep, counts):
    call("f2b_early_stop_rays", logit, int(logit_stride), dt, bounds, bounds.shape[0], weights, alphas, keep, counts, stream())


def count_scan(counts, n):
    bounds = dev_empty((n, 2), I32, counts)
    total = torch.zeros((1,), dtype=I32, device=counts.device)
    call("f2b_count_scan", counts, int(n), bounds, total, stream())
    return bounds, total


def compact_slots(keep, slot_bounds, new_bounds, rays_d, s_pts, s_dt, s_t, s_anchors, feat_slots, outs, feat_out):
    """outs = (pts, dirs, dt, t, anchors) destination arrays indexed by ``new_bounds``; bounds / rays_d may be chunk views."""
    call("f2b_compact_slots", keep, slot_bounds, new_bounds, slot_bounds.shape[0], rays_d, s_pts, s_dt, s_t, s_anchors,
         feat_slots, *outs, feat_out, stream())


def compact_samples(keep, old_bounds, new_bounds, n_kept, pts, dirs, dt, t, anchors, feat=None, feat_out=None):
    outs = (dev_empty((n_kept, 3), F32, pts), dev_empty((n_kept, 3), F32, pts), dev_empty((n_kept,), F32, pts),
            dev_empty((n_kept,), F32, pts), dev_empty((n_kept, 3), I32, pts))
    call("f2b_compact_samples", keep, old_bounds, new_bounds, old_bounds.shape[0], pts, dirs, dt, t, anchors, feat, *outs,
         feat_out, stream())
    return outs


def composite_fwd(logit, logit_stride, rgb, dt, t, bounds, bg):
    R, P = bounds.shape[0], dt.shape[0]
    colors, disp, depth = dev_empty((R, 3), F32, dt), dev_empty((R,), F32, dt), dev_empty((R,), F32, dt)
    weights = dev_empty((P,), F32, dt)
    call("f2b_composite_fwd", logit, int(logit_stride), rgb, dt, t, bounds, bg, R, colors, disp, depth, weights, stream())
    return colors, disp, depth, weights


def composite_bwd(logit, logit_stride, rgb, dt, t, bounds, bg, d_colors, d_disp, d_depth, d_weights, gs_progress,
                  d_logit, dlogit_stride):
    R, P = bounds.shape[0], dt.shape[0]
    d_rgb = dev_empty((P, 3), F32, dt)
    call("f2b_composite_bwd", logit, int(logit_stride), rgb, dt, t, bounds, bg, R, d_colors, d_disp, d_depth, d_weights,
         float(gs_progress), d_logit, int(dlogit_stride), d_rgb, stream())
    return d_rgb


# ------------------------------------------------------------------ reference free functions ----
class _FlexSum(torch.autograd.Function):
    @staticmethod
    def forward(ctx, val, idx_start_end):
        n, vec = idx_start_end.shape[0], (1 if val.dim() == 1 else val.shape[1])
        out = dev_empty((n,) if val.dim() == 1 else (n, vec), F32, val)
        call("f2b_flex_sum", val, vec, idx_start_end, n, out, stream())
        ctx.save_for_backward(idx_start_end)
        ctx.shape = val.shape
        return out

    @staticmethod
    def backward(ctx, g):
        (idx,) = ctx.saved_tensors
        lens = (idx[:, 1] - idx[:, 0]).long()
        return torch.repeat_interleave(g.contiguous(), lens, dim=0).reshape(ctx.shape), None


class _FlexAccumulateSum(torch.autograd.Function):
    @staticmethod
    def forward(ctx, val, idx_start_end, include_this):
        out = torch.empty_like(val)
        call("f2b_flex_accumulate_sum", val, idx_start_end, idx_start_end.shape[0], int(include_this), out, stream())
        ctx.save_for_backward(idx_start_end)
        ctx.include_this = include_this
        return out

    @staticmethod
    def backward(ctx, g):
        # reverse scan == total - forward scan of the gradient (FlexAccumulateSumBackwardKernel, FlexOps.cu:75-93)
        (idx,) = ctx.saved_tensors
        g = g.contiguous()
        fwd = torch.empty_like(g)
        call("f2b_flex_accumulate_sum", g, idx, idx.shape[0], int(not ctx.include_this), fwd, stream())
        tot = dev_empty((idx.shape[0],), F32, g)
        call("f2b_flex_sum", g, 1, idx, idx.shape[0], tot, stream())
        lens = (idx[:, 1] - idx[:, 0]).long()
        return torch.repeat_interleave(tot, lens) - fwd, None, None


class FlexOps:
    """FlexOps::Sum / FlexOps::AccumulateSum (src/Utils/CustomOps/FlexOps.h:15-16)."""

    @staticmethod
    def Sum(val, idx_start_end):
        return _FlexSum.apply(_chk(val.contiguous(), F32, "val"), _chk(idx_start_end.contiguous(), I32, "idx_start_end"))

    @staticmethod
    def AccumulateSum(val, idx_start_end, include_this):
        return _FlexAccumulateSum.apply(_chk(val.contiguous(), F32, "val"),
                                        _chk(idx_start_end.contiguous(), I32, "idx_start_end"), bool(include_this))


class _WeightVar(torch.autograd.Function):
    @staticmethod
    def forward(ctx, weights, idx_start_end):
        n = idx_start_end.shape[0]
        out = dev_empty((n,), F32, weights)
        call("f2b_weight_var_fwd", weights, idx_start_end, n, out, stream())
        ctx.save_for_backward(weights, idx_start_end)
        return out

    @staticmethod
    def backward(ctx, g):
        weights, idx = ctx.saved_tensors
        dw = torch.zeros_like(weights)
        call("f2b_weight_var_bwd", weights, idx, idx.shape[0], g.contiguous(), dw, stream())
        return dw, None


class _TruncExp(torch.autograd.Function):
    """TruncExp (CustomOps.cpp:9-18): exp forward, gradient with the exponent clamped to [-100, 5]."""

    @staticmethod
    def forward(ctx, x):
        ctx.save_for_backward(x)
        return torch.exp(x)

    @staticmethod
    def backward(ctx, g):
        (x,) = ctx.saved_tensors
        return g * torch.exp(x.clamp(-100.0, 5.0))


class CustomOps:
    """CustomOps::{WeightVar, ScatterIdx} and TruncExp with the reference's signatures."""

    @staticmethod
    def WeightVar(weights, idx_start_end):
        return _WeightVar.apply(_chk(weights.contiguous(), F32, "weights"),
                                _chk(idx_start_end.contiguous(), I32, "idx_start_end"))

    @staticmethod
    def ScatterIdx(n_all_pts, idx_start_end, emb_idx):
        return scatter_idx(n_all_pts, _chk(idx_start_end, I32, "idx_start_end"), _chk(emb_idx, I32, "emb_idx"))

    TruncExp = _TruncExp
