"""ctypes binding of the C ABI in include/f2nerf_b200.h (libf2nerf_b200.so, sm_100a only).

The product path has no CPU fallback: if the shared library is missing or does not load, importing
this module raises.  Tensors cross the boundary as raw device pointers (``Tensor.data_ptr()``) plus
sizes and the current CUDA stream; PyTorch is only the allocator / stream provider.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libf2nerf_b200.so")


class F2BError(RuntimeError):
    """Raised when a C-ABI call returns a negative status (message from f2b_last_error)."""


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"f2nerf_b200: CUDA extension {LIB_PATH} is missing — run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make`) first; there is no CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    lib.f2b_last_error.restype = ctypes.c_char_p
    return lib


lib = _load()

c_int, c_float, c_void_p, c_i64 = ctypes.c_int, ctypes.c_float, ctypes.c_void_p, ctypes.c_int64

# name -> argtypes (restype is always int).  Keep in the order of include/f2nerf_b200.h.
_P = c_void_p
SIGNATURES = {
    "f2b_abi_version": [],
    "f2b_device_info": [_P, _P],
    "f2b_sampler_count": [_P, c_int, _P, c_int, _P, _P, _P, c_int, c_float, c_float, c_float, c_int, c_int, c_int, _P, _P, _P, _P],
    "f2b_sampler_fill": [_P, c_int, _P, c_int, _P, _P, _P, c_int, c_float, c_float, c_float, c_int, c_int, _P, _P, _P, _P, _P, _P, _P, _P],
    "f2b_sampler_march": [_P, c_int, _P, c_int, _P, _P, _P, c_int, c_float, c_float, c_float, c_int, c_int, c_int, _P, _P, _P, _P,
                          _P, _P, _P, _P, _P],
    "f2b_sampler_march_bg": [_P, c_int, _P, c_int, _P, _P, _P, c_int, c_float, c_float, c_float, c_int, c_int, c_int, _P, _P, _P, _P,
                             _P, _P, _P, _P, _P],
    "f2b_sampler_gather": [_P, _P, c_int, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P],
    "f2b_edge_samples": [_P, _P, _P, _P, c_int, _P, _P, _P],
    "f2b_oct_mark_visit": [_P, c_int, _P, c_int, _P, _P, _P, _P, _P, _P, _P],
    "f2b_oct_update_stats": [_P, _P, _P, _P, _P, _P, c_int, _P],
    "f2b_hash_level_scales": [_P],
    "f2b_table_to_half": [_P, _P, c_i64, _P],
    "f2b_hash_fwd": [_P, _P, _P, c_int, c_int, _P, _P, c_int, c_int, _P, _P],
    "f2b_hash_fwd_levels": [_P, _P, _P, c_int, c_int, _P, _P, c_int, c_int, c_int, c_int, _P, _P],
    "f2b_hash_bwd": [_P, _P, c_int, c_int, _P, _P, c_int, c_int, _P, c_int, c_float, _P, _P],
    "f2b_hash_bwd_levels": [_P, _P, c_int, c_int, _P, _P, c_int, c_int, _P, c_int, c_float, _P, c_int, c_int, _P],
    "f2b_mlp_fwd": [_P, _P, c_int, c_int, _P, _P, _P],
    "f2b_mlp_fwd_f32": [_P, _P, c_int, c_int, _P, _P, _P, _P],
    "f2b_mlp_bwd": [_P, _P, _P, _P, c_int, c_int, _P, _P, _P],
    "f2b_field_shade_fwd": [_P, _P, _P, _P, _P, c_int, _P, _P, _P, _P],
    "f2b_shader_mlp_rgb_fwd": [_P, _P, c_int, _P, _P, _P, _P],
    "f2b_mlp_bwd2": [_P, _P, _P, _P, _P, c_int, c_int, _P, _P, _P],
    "f2b_field_bwd_scatter": [_P, _P, _P, c_int, _P, _P, c_int, _P, _P, _P, _P, c_int, c_int, c_float, _P, _P, _P],
    "f2b_mlp_fwd_v0": [_P, _P, c_int, c_int, _P, _P, _P],
    "f2b_mlp_bwd_v0": [_P, _P, _P, _P, c_int, c_int, _P, _P, _P],
    "f2b_mlp_fwd_tc": [_P, _P, c_int, c_int, _P, _P, _P],
    "f2b_mlp_bwd_tc": [_P, _P, _P, _P, c_int, c_int, _P, _P, _P],
    "f2b_field_fwd": [_P, _P, _P, c_int, c_int, _P, _P, _P, c_int, c_int, c_int, _P, _P, _P, _P],
    "f2b_field_fwd_slots": [_P, _P, _P, c_int, c_int, _P, _P, _P, c_int, _P, c_int, c_int, c_int, _P, _P, _P],
    "f2b_set_mlp_impl": [c_int],
    "f2b_get_mlp_impl": [],
    "f2b_cast_f32_to_f16": [_P, _P, c_i64, c_float, _P],
    "f2b_cast_f16_to_f32": [_P, _P, c_i64, c_float, _P],
    "f2b_sh_encode": [_P, c_int, c_int, _P, _P],
    "f2b_scatter_idx": [_P, _P, c_int, _P, _P],
    "f2b_shader_prep": [_P, _P, _P, _P, c_int, _P, _P],
    "f2b_shader_act": [_P, c_int, _P, _P],
    "f2b_shader_act_bwd": [_P, _P, c_int, c_float, _P, _P],
    "f2b_shader_prep_bwd": [_P, _P, _P, c_int, c_float, _P, _P, _P],
    "f2b_shader_prep_bwd_f16": [_P, _P, _P, _P, c_int, c_float, c_float, _P, _P, _P],
    "f2b_octree_proc": [_P, _P, _P, _P, c_int, c_int, c_int, _P, _P, _P, _P, _P, _P, _P],
    "f2b_octree_mark_invisible": [_P, c_int, _P, _P, _P, c_int, _P],
    "f2b_img2world_rays": [_P, _P, _P, _P, _P, c_int, _P, _P, _P],
    "f2b_gather_pixels": [_P, _P, _P, c_int, c_int, c_int, _P, _P],
    "f2b_adam_step": [_P, _P, _P, _P, c_i64, c_i64, ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.c_double,
                      ctypes.c_double, c_i64, _P, _P],
    "f2b_early_stop": [_P, c_int, _P, _P, c_int, _P, _P, _P, _P, _P, _P, _P],
    "f2b_early_stop_rays": [_P, c_int, _P, _P, c_int, _P, _P, _P, _P, _P],
    "f2b_count_scan": [_P, c_int, _P, _P, _P],
    "f2b_slot_bounds": [_P, c_int, c_int, c_int, _P, _P],
    "f2b_compact_slots": [_P, _P, _P, c_int, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P],
    "f2b_compact_samples": [_P, _P, _P, c_int, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P],
    "f2b_composite_fwd": [_P, c_int, _P, _P, _P, _P, _P, c_int, _P, _P, _P, _P, _P],
    "f2b_composite_bwd": [_P, c_int, _P, _P, _P, _P, _P, c_int, _P, _P, _P, _P, c_float, _P, c_int, _P, _P],
    "f2b_composite_act_bwd": [_P, c_int, _P, _P, _P, _P, _P, c_int, _P, _P, _P, _P, c_float, _P, c_float, _P, c_int, _P, _P],
    "f2b_flex_sum": [_P, c_int, _P, c_int, _P, _P],
    "f2b_flex_accumulate_sum": [_P, _P, c_int, c_int, _P, _P],
    "f2b_weight_var_fwd": [_P, _P, c_int, _P, _P],
    "f2b_weight_var_bwd": [_P, _P, c_int, _P, _P, _P],
    "f2b_render_fwd_fused": [_P, _P, _P, c_int, c_int, _P, _P, _P, _P, _P, _P, _P, _P, _P, c_int, c_int, _P, _P, _P, _P, _P, _P, _P, _P],
    "f2b_gather_kept_weights": [_P, _P, c_int, c_int, _P, _P],
}



class RenderArgs(ctypes.Structure):
    """``struct f2b_render`` (include/f2nerf_b200.h): the argument block of the per-phase launch sequences.  Field order and
    types mirror the header exactly (checked by tests/test_abi.py against sizeof on the C side)."""
    _P, _I, _F, _L = c_void_p, c_int, c_float, c_i64
    _fields_ = [
        ("tree_nodes", _P), ("n_nodes", _I), ("trans", _P), ("n_trans", _I), ("edge_pool", _P),
        ("near_t", _F), ("far_t", _F), ("sample_l", _F), ("scale_by_dis", _I), ("max_hits", _I), ("count_all_hits", _I),
        ("table16", _P), ("prim", _P), ("bias", _P), ("n_volumes", _I), ("local_size", _I),
        ("field_params", _P), ("n_field_params", _I), ("shader_params", _P), ("n_shader_params", _I),
        ("fparams16", _P), ("sparams16", _P),
        ("app_emb", _P), ("n_emb", _I),
        ("n_rays", _I), ("rays_o", _P), ("rays_d", _P), ("noise", _P), ("bg", _P),
        ("ray_emb_idx", _P),
        ("skip_march", _I),
        ("s_pts", _P), ("s_dt", _P), ("s_t", _P), ("s_anchors", _P), ("counts", _P), ("chunk_bounds", _P), ("slot_bounds", _P),
        ("first_oct_dis", _P), ("totals", _P),
        ("logit_s", _P), ("feat_s", _P), ("w0", _P), ("a0", _P), ("keep", _P), ("kept_counts", _P), ("new_bounds", _P), ("total_kept", _P),
        ("n_kept", _I), ("n_edge_pairs", _I),
        ("pts", _P), ("dirs", _P), ("dt", _P), ("t", _P), ("anchors", _P), ("feat_q", _P),
        ("edge_idx", _P), ("edge_coord", _P), ("e_pts", _P), ("e_anc", _P),
        ("pt_emb_idx", _P),
        ("logit", _P), ("mlp_in", _P), ("f_hidden", _P), ("edge32", _P), ("raw", _P), ("rgb", _P), ("s_hidden", _P),
        ("colors", _P), ("disparity", _P), ("depth", _P), ("weights", _P),
        ("d_colors", _P), ("d_disparity", _P), ("d_depth", _P), ("d_weights", _P), ("d_edge", _P),
        ("gs_progress", _F), ("shader_loss_scale", _F), ("field_loss_scale", _F), ("table_grad_mul", _F),
        ("d_logit", _P), ("d_raw", _P), ("d_in16", _P), ("d_scene16", _P), ("dfeat16", _P),
        ("d_sparams", _P), ("d_fparams", _P), ("d_table", _P), ("table_numel", _L), ("table_live", _L), ("d_app", _P),
        ("scatter_mode", _I),
        ("nonfinite", _P),
        ("stream", _P), ("side_stream", _P),
    ]

    def set(self, **kw):
        """Assign fields; tensors are passed by device pointer (None -> NULL), everything else as is."""
        for k, v in kw.items():
            if isinstance(v, torch.Tensor):
                if not v.is_contiguous():
                    raise ValueError(f"f2nerf_b200: tensor {k} crossing the C ABI must be contiguous")
                v = v.data_ptr()
            setattr(self, k, v)
        return self


SIGNATURES["f2b_render_sizeof"] = []
for _name in ("f2b_render_phase1", "f2b_render_phase2_fwd", "f2b_render_bwd", "f2b_render_grad_finalize"):
    SIGNATURES[_name] = [ctypes.POINTER(RenderArgs)]
lib.f2b_render_sizeof.restype = c_int
lib.f2b_render_sizeof.argtypes = []
if lib.f2b_render_sizeof() != ctypes.sizeof(RenderArgs):
    raise ImportError(f"f2nerf_b200: struct f2b_render is {lib.f2b_render_sizeof()} bytes in the library but "
                      f"{ctypes.sizeof(RenderArgs)} in the binding — header / _lib.py out of step")

for _name, _args in SIGNATURES.items():
    _fn = getattr(lib, _name)          # AttributeError here == header/library mismatch: fail loudly
    _fn.argtypes = _args
    _fn.restype = c_int


def ptr(t):
    """Device (or host) pointer of a contiguous tensor, None -> NULL."""
    if t is None:
        return None
    if isinstance(t, torch.Tensor):
        if not t.is_contiguous():
            raise ValueError("f2nerf_b200: tensor crossing the C ABI must be contiguous")
        return t.data_ptr()
    return t


def stream():
    return torch.cuda.current_stream().cuda_stream


# The field-MLP backward and the hash scatter as one kernel (f2b_field_bwd_scatter); F2B_FIELD_BWD_SCATTER=0 restores the
# two-kernel sequence (f2b_mlp_bwd2 -> fp16 dL/dfeatures in memory -> f2b_hash_bwd) for A/B runs.  The data-parallel level-slab
# scatter always runs the two-kernel sequence.
FIELD_BWD_SCATTER = os.environ.get("F2B_FIELD_BWD_SCATTER", "1") != "0"

# kernels launched per entry point (for bench.py's gpu_launches claim; memsets are not counted)
KERNELS_PER_CALL = {"f2b_render_sizeof": 0, "f2b_render_phase1": 7, "f2b_render_phase2_fwd": 10,
                    "f2b_render_bwd": 5 if FIELD_BWD_SCATTER else 8, "f2b_render_grad_finalize": 2, "f2b_field_bwd_scatter": 1,
                    "f2b_sampler_count": 2, "f2b_sampler_march": 2, "f2b_sampler_march_bg": 2, "f2b_early_stop": 2, "f2b_hash_level_scales": 1, "f2b_device_info": 0,
                    "f2b_abi_version": 0, "f2b_set_mlp_impl": 0, "f2b_get_mlp_impl": 0}
LAUNCHES = 0      # running count of product kernels launched through this binding
TRACE = None      # set to a list to record (name, start_event, end_event, int_args) per call (bench.py)


def call(name, *args):
    """Invoke a C-ABI entry point; tensors are passed by pointer; raises F2BError on failure."""
    global LAUNCHES
    fn = getattr(lib, name)
    conv = [ptr(a) if isinstance(a, torch.Tensor) or a is None else (ctypes.byref(a) if isinstance(a, ctypes.Structure) else a)
            for a in args]
    if TRACE is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        rc = fn(*conv)
        e1.record()
        TRACE.append((name, e0, e1, [a for a in args if isinstance(a, int) and not isinstance(a, bool)]))
    else:
        rc = fn(*conv)
    if rc != 0:
        raise F2BError(f"{name} -> {rc}: {lib.f2b_last_error().decode()}")
    LAUNCHES += KERNELS_PER_CALL.get(name, 1)
    return rc
