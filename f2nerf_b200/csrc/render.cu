// render.cu — the per-batch launch sequences of the fused Renderer::Render pipeline behind single C-ABI calls
// (f2b_render_phase1 / _phase2_fwd / _bwd / _grad_finalize, include/f2nerf_b200.h).
//
// Why: measured on B200 (profiles/r02_timeline.md) the step spent ~0.8 ms with the GPU idle behind the one host sync of
// Renderer::Render — a Python host needs ~130 foreign calls / allocator calls to enqueue the second half of the step, and
// the short kernels right after the sync finish faster than it can launch them.  The sequences are fixed, so they live here:
// one foreign call per phase, the kernels back to back.  No new arithmetic: every launch goes through the entry points
// declared earlier in the header (same kernels, same order, same streams as f2nerf_b200/renderer.py used to issue one by one);
// the only kernels of this file are the gradient un-scaling + finiteness flags that replace ~10 ATen passes.
#include "common.cuh"
#include <stdlib.h>

namespace f2b {

// d_sparams *= 1/s_scale, d_fparams *= 1/f_scale (tensor / python-scalar in ATen multiplies by the reciprocal; the scales are
// powers of two), flags[0] |= nonfinite(d_sparams) | nonfinite(d_app), flags[1] |= nonfinite(d_fparams)
__global__ void finalize_small_kernel(float* __restrict__ d_sparams, int n_s, float inv_s, float* __restrict__ d_fparams, int n_f,
                                      float inv_f, const float* __restrict__ d_app, int n_app, int* __restrict__ flags) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  int bad_s = 0, bad_f = 0;
  if (i < n_s) { const float v = d_sparams[i] * inv_s; d_sparams[i] = v; bad_s |= !isfinite(v); }
  if (i < n_f) { const float v = d_fparams[i] * inv_f; d_fparams[i] = v; bad_f |= !isfinite(v); }
  if (d_app && i < n_app) bad_s |= !isfinite(d_app[i]);
  if (__any_sync(0xffffffffu, bad_s) && (threadIdx.x & 31) == 0) atomicOr(flags, 1);
  if (__any_sync(0xffffffffu, bad_f) && (threadIdx.x & 31) == 0) atomicOr(flags + 1, 1);
}
// flags[1] |= nonfinite(d_table[0:live])   (the field MLP's dL/dinput reaches every table entry its samples touch)
__global__ void finalize_table_kernel(const float4* __restrict__ g, int64_t n4, int* __restrict__ flags) {
  int bad = 0;
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n4; i += int64_t(gridDim.x) * blockDim.x) {
    const float4 v = g[i];
    bad |= !(isfinite(v.x) && isfinite(v.y) && isfinite(v.z) && isfinite(v.w));
  }
  if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) atomicOr(flags + 1, 1);
}

}  // namespace f2b

using namespace f2b;

#define F2B_TRY(expr)            \
  do {                           \
    const int rc_ = (expr);      \
    if (rc_ != F2B_OK) return rc_; \
  } while (0)
#define F2B_CUDA(expr, what)                                                                          \
  do {                                                                                                \
    const cudaError_t e_ = (expr);                                                                    \
    if (e_ != cudaSuccess) { set_error("%s: CUDA error %d (%s)", what, (int)e_, cudaGetErrorString(e_)); return F2B_ECUDA; } \
  } while (0)

static inline char* off(void* p, int64_t bytes) { return reinterpret_cast<char*>(p) + bytes; }

static bool field_bwd_scatter_on() {
  static int on = -1;
  if (on < 0) { const char* e = getenv("F2B_FIELD_BWD_SCATTER"); on = !(e && atoi(e) == 0); }
  return on != 0;
}

extern "C" int f2b_render_sizeof(void) { return (int)sizeof(f2b_render); }       // binding self-check (layout drift = refuse to load)

extern "C" int f2b_render_phase1(const f2b_render* r) {
  F2B_REQUIRE(r, "f2b_render_phase1: null argument block");
  if (r->n_rays <= 0) return F2B_OK;
  const int S = F2B_MAX_SAMPLE_PER_RAY;
  if (!r->skip_march) {
    F2B_TRY(f2b_sampler_march(r->tree_nodes, r->n_nodes, r->trans, r->n_trans, r->rays_o, r->rays_d, r->noise, r->n_rays, r->near_t,
                              r->far_t, r->sample_l, r->scale_by_dis, r->max_hits, r->count_all_hits, r->s_pts, r->s_dt, r->s_t,
                              r->s_anchors, r->counts, r->chunk_bounds, r->totals, r->first_oct_dis, r->stream));
    F2B_TRY(f2b_slot_bounds(r->counts, r->n_rays, S, 0, r->slot_bounds, r->stream));
  }
  F2B_TRY(f2b_cast_f32_to_f16(r->field_params, r->fparams16, r->n_field_params, 1.f, r->stream));
  F2B_TRY(f2b_field_fwd_slots(r->table16, r->prim, r->bias, r->n_volumes, r->local_size, r->fparams16, r->s_pts, r->s_anchors, 2,
                              r->counts, r->n_rays, S, 1, r->logit_s, r->feat_s, r->stream));
  F2B_TRY(f2b_early_stop_rays(r->logit_s, 1, r->s_dt, r->slot_bounds, r->n_rays, r->w0, r->a0, r->keep, r->kept_counts, r->stream));
  F2B_CUDA(cudaMemsetAsync(r->total_kept, 0, sizeof(int), as_stream(r->stream)), "f2b_render_phase1");
  return f2b_count_scan(r->kept_counts, r->n_rays, r->new_bounds, r->total_kept, r->stream);
}

extern "C" int f2b_render_phase2_fwd(const f2b_render* r) {
  F2B_REQUIRE(r, "f2b_render_phase2_fwd: null argument block");
  if (r->n_rays <= 0) return F2B_OK;
  const int64_t nk = r->n_kept, ne = 2 * int64_t(r->n_edge_pairs);
  F2B_TRY(f2b_compact_slots(r->keep, r->slot_bounds, r->new_bounds, r->n_rays, r->rays_d, r->s_pts, r->s_dt, r->s_t, r->s_anchors,
                            r->feat_s, r->pts, r->dirs, r->dt, r->t, r->anchors, r->feat_q, r->stream));
  if (ne > 0) {                                                    // TV-loss edge points (Renderer.cpp:153-166)
    F2B_TRY(f2b_edge_samples(r->edge_pool, r->trans, r->edge_idx, r->edge_coord, r->n_edge_pairs, r->e_pts, r->e_anc, r->stream));
    F2B_TRY(f2b_hash_fwd(r->table16, r->prim, r->bias, r->n_volumes, r->local_size, r->e_pts, r->e_anc, 1, (int)ne,
                         off(r->feat_q, nk * 64), r->stream));
  }
  const bool emb = r->app_emb && r->ray_emb_idx;
  if (emb && nk > 0) F2B_TRY(f2b_scatter_idx(r->new_bounds, r->ray_emb_idx, r->n_rays, r->pt_emb_idx, r->stream));
  F2B_TRY(f2b_cast_f32_to_f16(r->field_params, r->fparams16, r->n_field_params, 1.f, r->stream));
  F2B_TRY(f2b_cast_f32_to_f16(r->shader_params, r->sparams16, r->n_shader_params, 1.f, r->stream));
  F2B_TRY(f2b_field_shade_fwd(r->feat_q, r->fparams16, r->dirs, emb ? r->app_emb : nullptr, emb ? r->pt_emb_idx : nullptr, (int)nk,
                              r->logit, r->mlp_in, r->f_hidden, r->stream));
  if (ne > 0)
    F2B_TRY(f2b_mlp_fwd_f32(off(r->feat_q, nk * 64), r->fparams16, 0, (int)ne, r->edge32, nullptr,
                            r->f_hidden ? off(r->f_hidden, nk * 128) : nullptr, r->stream));
  F2B_TRY(f2b_shader_mlp_rgb_fwd(r->mlp_in, r->sparams16, (int)nk, r->raw, r->rgb, r->s_hidden, r->stream));
  return f2b_composite_fwd(r->logit, 1, r->rgb, r->dt, r->t, r->new_bounds, r->bg, r->n_rays, r->colors, r->disparity, r->depth,
                           r->weights, r->stream);
}

extern "C" int f2b_render_bwd(const f2b_render* r) {
  F2B_REQUIRE(r, "f2b_render_bwd: null argument block");
  // f_hidden / s_hidden NULL: the forward saved no hidden activations, f2b_mlp_bwd2 rebuilds them (recompute, tcgen05 only)
  const int64_t nk = r->n_kept, ne = 2 * int64_t(r->n_edge_pairs), nq = nk + ne;
  cudaStream_t st = as_stream(r->stream), side = as_stream(r->side_stream);
  const bool emb = r->app_emb && r->ray_emb_idx;
  // scatter_mode 0: f2b_field_bwd_scatter unless F2B_FIELD_BWD_SCATTER=0 (the two-kernel sequence through dfeat16, for A/B runs)
  const bool fused = r->scatter_mode == 0 && field_bwd_scatter_on();
  F2B_CUDA(cudaMemsetAsync(r->d_sparams, 0, sizeof(float) * r->n_shader_params, st), "f2b_render_bwd");
  F2B_CUDA(cudaMemsetAsync(r->d_fparams, 0, sizeof(float) * r->n_field_params, st), "f2b_render_bwd");
  F2B_CUDA(cudaMemsetAsync(r->d_table, 0, sizeof(float) * r->table_numel, st), "f2b_render_bwd");
  F2B_CUDA(cudaMemsetAsync(r->nonfinite, 0, 2 * sizeof(int), st), "f2b_render_bwd");
  if (emb) F2B_CUDA(cudaMemsetAsync(r->d_app, 0, sizeof(float) * 16 * r->n_emb, st), "f2b_render_bwd");
  if (ne > 0) {                                                    // dL/d edge features -> the field MLP's fp16, loss-scaled dL/dout rows
    if (r->d_edge) F2B_TRY(f2b_cast_f32_to_f16(r->d_edge, off(r->d_scene16, nk * 32), ne * 16, r->field_loss_scale, r->stream));
    else F2B_CUDA(cudaMemsetAsync(off(r->d_scene16, nk * 32), 0, ne * 32, st), "f2b_render_bwd");
  }
  if (nk > 0) {
    F2B_TRY(f2b_composite_act_bwd(r->logit, 1, r->rgb, r->dt, r->t, r->new_bounds, r->bg, r->n_rays, r->d_colors, r->d_disparity,
                                  r->d_depth, r->d_weights, r->gs_progress, r->raw, r->shader_loss_scale, r->d_logit, 1, r->d_raw,
                                  r->stream));
    F2B_TRY(f2b_mlp_bwd2(r->d_raw, r->mlp_in, r->s_hidden, r->s_hidden ? off(r->s_hidden, nk * 128) : nullptr, r->sparams16, 1, (int)nk, r->d_in16, r->d_sparams,
                         r->stream));
    F2B_TRY(f2b_shader_prep_bwd_f16(r->d_in16, r->d_logit, r->new_bounds, emb ? r->ray_emb_idx : nullptr, r->n_rays,
                                    1.f / r->shader_loss_scale, r->field_loss_scale, r->d_scene16, emb ? r->d_app : nullptr, r->stream));
    if (!fused) F2B_TRY(f2b_mlp_bwd2(r->d_scene16, r->feat_q, r->f_hidden, nullptr, r->fparams16, 0, (int)nk, r->dfeat16, r->d_fparams, r->stream));
  }
  if (fused)                                                       // field MLP backward + scatter of both segments, one launch
    return f2b_field_bwd_scatter(r->d_scene16, r->feat_q, r->fparams16, (int)nk, r->pts, r->anchors, (int)ne, r->e_pts, r->e_anc, r->prim,
                                 r->bias, r->n_volumes, r->local_size, r->table_grad_mul, r->d_fparams, r->d_table, r->stream);
  if (ne > 0)
    F2B_TRY(f2b_mlp_bwd2(off(r->d_scene16, nk * 32), off(r->feat_q, nk * 64), r->f_hidden ? off(r->f_hidden, nk * 128) : nullptr, nullptr, r->fparams16, 0, (int)ne,
                         off(r->dfeat16, nk * 64), r->d_fparams, r->stream));
  if (r->scatter_mode != 0) return F2B_OK;
  // the scatter (L2 reductions) on the side stream behind the dense chain, joined before returning
  cudaEvent_t fork, join;
  F2B_CUDA(cudaEventCreateWithFlags(&fork, cudaEventDisableTiming), "f2b_render_bwd");
  F2B_CUDA(cudaEventCreateWithFlags(&join, cudaEventDisableTiming), "f2b_render_bwd");
  cudaEventRecord(fork, st);
  cudaStreamWaitEvent(side, fork, 0);
  int rc = F2B_OK;
  if (nk > 0)
    rc = f2b_hash_bwd(r->prim, r->bias, r->n_volumes, r->local_size, r->pts, r->anchors, 3, (int)nk, r->dfeat16, 1, r->table_grad_mul,
                      r->d_table, r->side_stream);
  if (rc == F2B_OK && ne > 0)
    rc = f2b_hash_bwd(r->prim, r->bias, r->n_volumes, r->local_size, r->e_pts, r->e_anc, 1, (int)ne, off(r->dfeat16, nk * 64), 1,
                      r->table_grad_mul, r->d_table, r->side_stream);
  cudaEventRecord(join, side);
  cudaStreamWaitEvent(st, join, 0);
  cudaEventDestroy(fork);
  cudaEventDestroy(join);
  (void)nq;
  return rc;
}

extern "C" int f2b_render_grad_finalize(const f2b_render* r) {
  F2B_REQUIRE(r && r->d_sparams && r->d_fparams && r->nonfinite, "f2b_render_grad_finalize: null pointer");
  const bool emb = r->app_emb && r->ray_emb_idx;
  const int n_app = emb ? 16 * r->n_emb : 0;
  int n = r->n_shader_params > r->n_field_params ? r->n_shader_params : r->n_field_params;
  if (n_app > n) n = n_app;
  finalize_small_kernel<<<div_up(n, 256), 256, 0, as_stream(r->stream)>>>(r->d_sparams, r->n_shader_params, 1.f / r->shader_loss_scale,
                                                                           r->d_fparams, r->n_field_params, 1.f / r->field_loss_scale,
                                                                           emb ? r->d_app : nullptr, n_app, r->nonfinite);
  if (r->d_table && r->table_live >= 4) {
    int sms = 148;
    f2b_device_info(&sms, nullptr);
    finalize_table_kernel<<<sms * 4, 256, 0, as_stream(r->stream)>>>(reinterpret_cast<const float4*>(r->d_table), r->table_live / 4,
                                                                     r->nonfinite);
  }
  return check_launch("f2b_render_grad_finalize");
}
