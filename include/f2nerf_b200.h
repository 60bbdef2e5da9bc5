/* f2nerf_b200.h — C ABI of the B200-native (sm_100a) F2-NeRF per-ray rendering hot path.
 *
 * Every entry point takes plain device pointers + sizes + a cudaStream_t (as void*), never
 * allocates, never retains a pointer past the call, never throws.  Return value: 0 on success,
 * negative F2B_E* on error (message via f2b_last_error()).  No torch types cross this boundary.
 *
 * Each function names the reference interface (file:line under Totoro97/f2-nerf @98f0daa) it
 * replaces.  Byte layouts of the octree blobs are the reference's own (PersSampler.h:15-37):
 *   TreeNode  64 B : center f32x3 @0, side_len f32 @12, parent i32 @16, childs i32x8 @20,
 *                    is_leaf u8 @52, trans_idx i32 @56
 *   TransInfo 544 B: w2xz[12] row-major 2x4 f32 @0, weight row-major 3x12 f32 @384,
 *                    center f32x3 @528, dis_summary f32 @540
 *   EdgePool  64 B : t_idx_a i32 @0, t_idx_b i32 @4, center f32x3 @8, dir_0 f32x3 @20, dir_1 f32x3 @32
 */
#ifndef F2NERF_B200_H
#define F2NERF_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define F2B_OK            0
#define F2B_EINVAL      (-1)
#define F2B_ECUDA       (-2)
#define F2B_EUNSUPPORTED (-3)

#define F2B_N_LEVELS    16
#define F2B_N_CHANNELS   2
#define F2B_N_PROS      12
#define F2B_MAX_SAMPLE_PER_RAY 1024
#define F2B_MLP_WIDTH   64
#define F2B_MLP_IN      32
#define F2B_MLP_OUT_PAD 16

const char* f2b_last_error(void);
int  f2b_abi_version(void);
/* SM count / L2 bytes of the current device (grid sizing, bench reporting). */
int  f2b_device_info(int* sm_count, int* l2_bytes);

/* ------------------------------------------------------------------------------------------
 * Sampler  — replaces PersSampler::GetSamples (src/PtsSampler/PersSampler.cu:317-434):
 * FindRayOctreeIntersectionKernel<false/true> (:53-152) + RayMarchKernel<false/true> (:189-314)
 * are fused into one traverse-and-march kernel run twice (count, fill); the host syncs once
 * (to size the outputs) instead of twice, and no hit list is materialised in HBM.
 * rays_d must already be unit length (the reference normalises with ATen at :319).
 * rays_noise has F2B_MAX_SAMPLE_PER_RAY + n_rays + 10 floats, already scaled by fineness (:373-381).
 * ------------------------------------------------------------------------------------------ */
/* Pass 1: per-ray sample counts -> exclusive/inclusive bounds (reference: cumsum at :395),
 * totals[0] = n_all_pts, totals[1] = octree hits: with count_all_hits != 0 the exact n_all_oct_intersect of
 * :353 (the traversal is run to exhaustion — only feeds the informational sampled_oct_per_ray EMA, :378),
 * otherwise the hits the march actually consumed. */
int f2b_sampler_count(const void* tree_nodes, int n_nodes, const void* trans, int n_trans,
                      const float* rays_o, const float* rays_d, const float* rays_noise, int n_rays,
                      float near, float far, float sample_l, int scale_by_dis,
                      int max_oct_intersect_per_ray, int count_all_hits,
                      int* ray_counts /* [n_rays] caller-owned scratch */,
                      int* pts_idx_bounds /* [n_rays,2] out */, int* totals /* [2] out */,
                      void* stream);
/* Pass 2: emit samples.  anchors is [P,3] i32: [:,0]=trans_idx, [:,1]=node idx, [:,2]=0
 * (the reference leaves [:,2] uninitialised, PersSampler.cu:284-285). */
int f2b_sampler_fill(const void* tree_nodes, int n_nodes, const void* trans, int n_trans,
                     const float* rays_o, const float* rays_d, const float* rays_noise, int n_rays,
                     float near, float far, float sample_l, int scale_by_dis,
                     int max_oct_intersect_per_ray, const int* pts_idx_bounds,
                     float* pts /* [P,3] warped */, float* dirs /* [P,3] */, float* dt /* [P] */,
                     float* t /* [P] */, int* anchors /* [P,3] */, float* first_oct_dis /* [n_rays] */,
                     void* stream);
/* One-pass variant (what the host mirrors use): the march runs ONCE, each ray writing into its own scratch slot
 * of F2B_MAX_SAMPLE_PER_RAY samples (caller-owned scratch: s_pts [R*1024,3] f32, s_dt/s_t [R*1024] f32,
 * s_anchors [R*1024,2] i32 = trans_idx,node), then f2b_sampler_gather packs the slots into the reference's
 * compact ray-ordered layout (a 28 B/sample copy instead of a second traverse-and-march).  Outputs are
 * bit-identical to f2b_sampler_count + f2b_sampler_fill. */
int f2b_sampler_march(const void* tree_nodes, int n_nodes, const void* trans, int n_trans,
                      const float* rays_o, const float* rays_d, const float* rays_noise, int n_rays,
                      float near, float far, float sample_l, int scale_by_dis,
                      int max_oct_intersect_per_ray, int count_all_hits,
                      float* s_pts, float* s_dt, float* s_t, int* s_anchors,
                      int* ray_counts /* [n_rays] */, int* pts_idx_bounds /* [n_rays,2] out */, int* totals /* [2] out */,
                      float* first_oct_dis /* [n_rays] out */, void* stream);
/* The same march compiled for <= 64 registers per thread (identical arithmetic and results): for the software-pipelined march of
 * the NEXT batch, which runs on a side stream under this batch's backward and must leave the register file to the kernels it
 * shares the SMs with. */
int f2b_sampler_march_bg(const void* tree_nodes, int n_nodes, const void* trans, int n_trans,
                      const float* rays_o, const float* rays_d, const float* rays_noise, int n_rays,
                      float near, float far, float sample_l, int scale_by_dis,
                      int max_oct_intersect_per_ray, int count_all_hits,
                      float* s_pts, float* s_dt, float* s_t, int* s_anchors,
                      int* ray_counts /* [n_rays] */, int* pts_idx_bounds /* [n_rays,2] out */, int* totals /* [2] out */,
                      float* first_oct_dis /* [n_rays] out */, void* stream);
int f2b_sampler_gather(const float* rays_d, const int* pts_idx_bounds, int n_rays,
                       const float* s_pts, const float* s_dt, const float* s_t, const int* s_anchors,
                       float* pts, float* dirs, float* dt, float* t, int* anchors, void* stream);
/* GetEdgeSamplesKernel (PersSampler.cu:436-452). */
int f2b_edge_samples(const void* edge_pool, const void* trans, const int* edge_idx,
                     const float* edge_coord /* [n,2] */, int n_pts,
                     float* out_pts /* [n,2,3] */, int* out_idx /* [n,2] */, void* stream);
/* MarkVistNodeKernel (PersSampler.cu:475-526). oct_idx has element stride oct_stride (3 for anchors[:,1]). */
int f2b_oct_mark_visit(const int* pts_idx_bounds, int n_rays, const int* oct_idx, int oct_stride,
                       const float* weights, const float* alphas,
                       int* vote_weight, int* vote_alpha, int* visit_mark, int* visit_cnt,
                       void* stream);
/* The ATen stat update + MarkInvalidNodes (PersSampler.cu:579-603) in one kernel. */
int f2b_oct_update_stats(const int* vote_weight, const int* vote_alpha, const int* visit_mark,
                         int* weight_stats, int* alpha_stats, void* tree_nodes, int n_nodes,
                         void* stream);

/* ------------------------------------------------------------------------------------------
 * Field — replaces Hash3DAnchored::AnchoredQuery (src/Field/Hash3DAnchored.cpp:84-99),
 * Hash3DAnchoredFunction::forward/backward (Hash3DAnchored.cu:160-233) and TCNNWP::Query
 * (TCNNWP.cpp:102-243, tiny-cuda-nn FullyFusedMLP<half,64>).
 * table_f16: the fp16 shadow of feat_pool_ ([pool_size,2] halves); level l starts at half
 * element l*local_size (the reference's overlapping-level quirk, Hash3DAnchored.cu:37).
 * ------------------------------------------------------------------------------------------ */
/* The 16 per-level scales exp2f(7*l/15+3) exactly as the device computes them
 * (Hash3DAnchored.cu:29; MUFU.EX2 is not reproducible on a CPU, so the oracle takes these). */
int f2b_hash_level_scales(float* scales16_host);
/* fp32 master table -> fp16 shadow (Hash3DAnchored.cu:186 does this on every call). */
int f2b_table_to_half(const float* table_f32, void* table_f16, int64_t n, void* stream);
/* Encode: pts are the sampler's warped coordinates (the (p+1)/2 of Hash3DAnchored.cpp:91 is fused).
 * vol = anchors[:,0] with element stride vol_stride.  out: [P,32] fp16 (level-major, 2 ch). */
int f2b_hash_fwd(const void* table_f16, const int* prim_pool, const float* bias_pool,
                 int n_volumes, int local_size,
                 const float* pts, const int* vol, int vol_stride, int n_pts,
                 void* out_f16, void* stream);
/* f2b_hash_fwd for levels [level_lo, level_lo + n_levels) only: writes columns 2*l, 2*l+1 of those levels into out [P,32] and
 * leaves the rest untouched (per-level attribution of the encode's cost, partial refreshes). */
int f2b_hash_fwd_levels(const void* table_f16, const int* prim_pool, const float* bias_pool,
                        int n_volumes, int local_size, const float* pts, const int* vol,
                        int vol_stride, int n_pts, int level_lo, int n_levels, void* out_f16, void* stream);
/* Backward: grad_feat [P,32] (fp16 when grad_is_f16, else fp32; dL/d encoded features), each value
 * multiplied by grad_mul (e.g. 1/loss_scale), scattered into grad_table [pool_size,2] fp32 (zeroed by
 * the caller) with red.global.add.v2.f32 — instead of the reference's fp16 atomicAdd(__half2) of
 * grad*128 and a later /128 (Hash3DAnchored.cu:81-155,199-233). */
int f2b_hash_bwd(const int* prim_pool, const float* bias_pool, int n_volumes, int local_size,
                 const float* pts, const int* vol, int vol_stride, int n_pts,
                 const void* grad_feat, int grad_is_f16, float grad_mul,
                 float* grad_table, void* stream);
/* f2b_hash_bwd restricted to levels [level_lo, level_lo + n_levels), n_levels a power of two.  Level l only writes floats
 * [l*local_size, (l+2)*local_size) of grad_table, so a data-parallel host can launch level groups top-down and all-reduce each
 * finished slab (everything from float (level_lo+1)*local_size upwards) while the lower groups still scatter. */
int f2b_hash_bwd_levels(const int* prim_pool, const float* bias_pool, int n_volumes, int local_size,
                        const float* pts, const int* vol, int vol_stride, int n_pts,
                        const void* grad_feat, int grad_is_f16, float grad_mul, float* grad_table,
                        int level_lo, int n_levels, void* stream);

/* MLP (no biases, ReLU hidden, linear out padded to 16): params_f16 = [W0 64xin | (W_h 64x64)*n_hidden_matmuls | W_out 16x64],
 * each row-major [out][in] (fully_fused_mlp.cu:654-677).  in: [P,32] fp16.  out: [P,16] fp16.
 * hidden_save: nullable, [(n_hidden_matmuls+1), P, 64] fp16 forward activations for backward. */
int f2b_mlp_fwd(const void* in_f16, const void* params_f16, int n_hidden_matmuls, int n_pts,
                void* out_f16, void* hidden_save_f16, void* stream);
/* Same network with the output widened to fp32 in the epilogue — what TCNNWP::Query returns
 * (`feat...to(torch::kFloat32)`, TCNNWP.cpp:112).  out_f32 [P,16] and/or out_f16 [P,16]; with the tcgen05
 * implementation either may be NULL (not both), the CUDA-core twin needs out_f16. */
int f2b_mlp_fwd_f32(const void* in_f16, const void* params_f16, int n_hidden_matmuls, int n_pts,
                    float* out_f32, void* out_f16, void* hidden_save_f16, void* stream);
/* Backward: dL/dout [P,16] fp16 (already multiplied by loss_scale) -> dL/din [P,32] fp16 (nullable),
 * dL/dparams fp32 (same layout as params, accumulated in fp32; caller zeroes), both still scaled. */
int f2b_mlp_bwd(const void* dout_f16, const void* in_f16, const void* hidden_save_f16,
                const void* params_f16, int n_hidden_matmuls, int n_pts,
                void* din_f16, float* dparams_f32, void* stream);
/* fp32 -> fp16 elementwise with optional scale (identity encoding / loss-scale casts, TCNNWP.cpp:111,168). */
int f2b_cast_f32_to_f16(const float* src, void* dst, int64_t n, float scale, void* stream);
int f2b_cast_f16_to_f32(const void* src, float* dst, int64_t n, float scale, void* stream);

/* Fused Hash3DAnchored::AnchoredQuery (Hash3DAnchored.cpp:84-99): hash encode + tcgen05 MLP(32->64->16) in one
 * kernel; the encoded features reach HBM only through feat_save (backward needs them).
 * logit_only != 0: the no-grad early-stop pass — out is [P] fp32 (channel 0 only); feat_save optional, no hidden_save.
 * otherwise out is [P,16] fp32 (fp16-rounded values, as TCNNWP::Query returns); feat_save [P,32] fp16 and
 * hidden_save [P,64] fp16 are optional. */
int f2b_field_fwd(const void* table_f16, const int* prim_pool, const float* bias_pool, int n_volumes,
                  int local_size, const void* mlp_params_f16, const float* pts, const int* vol, int vol_stride,
                  int n_pts, int logit_only, float* out_f32, void* feat_save_f16, void* hidden_save_f16,
                  void* stream);

/* The same kernel over the one-pass march's scratch slots: ray r owns slots [r*slot_size, r*slot_size+ray_counts[r])
 * of slot_pts / slot_vol (slot_size a multiple of 128; tiles past a ray's count are skipped whole).  Outputs use the
 * same slot indexing.  Lets the early-stop pass of Renderer::Render (Renderer.cpp:107-126) start right behind the
 * march without the cumsum / host sync / gather that PersSampler::GetSamples performs (PersSampler.cu:395-398). */
int f2b_field_fwd_slots(const void* table_f16, const int* prim_pool, const float* bias_pool, int n_volumes,
                        int local_size, const void* mlp_params_f16, const float* slot_pts, const int* slot_vol,
                        int vol_stride, const int* ray_counts, int n_rays, int slot_size, int logit_only,
                        float* out_f32, void* feat_save_f16, void* stream);

/* Field MLP on already-encoded features with the shading-feature assembly fused into its epilogue (the fp32 [P,16]
 * scene_feat tensor, `ones_like`/`cat`/ScatterAdd of Renderer.cpp:179-187 and the SH encode + cast of SHShader.cpp:23-26
 * never materialise): logit[p] = out[p,0]; mlp_in[p] = fp16([1, out[p,1:16]] + app_emb[pt_emb_idx[p]] | SH4(dirs[p])).
 * tcgen05 implementation only (F2B_EUNSUPPORTED with the CUDA-core twin selected). */
int f2b_field_shade_fwd(const void* feat_f16 /* [P,32] */, const void* field_params_f16, const float* dirs /* [P,3] */,
                        const float* app_emb /* [n_emb,16] or NULL */, const int* pt_emb_idx /* [P] or NULL */, int n_pts,
                        float* logit /* [P] */, void* mlp_in_f16 /* [P,32] */, void* hidden_save_f16 /* [P,64] or NULL */,
                        void* stream);
/* Shader MLP with the colour activation of SHShader.cpp:27-28 in its epilogue: raw [P,16] fp16 and
 * rgb [P,3] = (1 + 2e-3) * sigmoid(raw[:, :3]) - 1e-3.  tcgen05 implementation only. */
int f2b_shader_mlp_rgb_fwd(const void* mlp_in_f16, const void* shader_params_f16, int n_pts, void* raw_f16, float* rgb,
                           void* hidden_save_f16 /* [2,P,64] or NULL */, void* stream);
/* f2b_mlp_bwd on a row range of a larger saved batch: the two activation layers are passed as separate pointers
 * (hidden1 NULL when n_hidden_matmuls == 0).  dparams is accumulated into, like f2b_mlp_bwd.
 * hidden0 == NULL (tcgen05 implementation only): the forward saved nothing — the kernel rebuilds the tile's hidden
 * activations from in_f16 on the tensor pipe (bit-identical to what the forward would have saved) before the backward;
 * 96 B read + 64 B written per sample instead of 224 / 352 + 64 (and the forward does not write 128 / 256 B). */
int f2b_mlp_bwd2(const void* dout_f16, const void* in_f16, const void* hidden0_f16, const void* hidden1_f16,
                 const void* params_f16, int n_hidden_matmuls, int n_pts, void* din_f16, float* dparams_f32, void* stream);
/* Field-MLP backward and hash-table scatter in one kernel: f2b_mlp_bwd2(dout, in, NULL, NULL, params, 0, ...) followed by
 * f2b_hash_bwd of its fp16 dL/dinput, without the dL/dinput rows ever reaching memory.  Rows [0, n_kept) of dout_f16 [.,16] /
 * in_f16 [.,32] are the samples at pts [n_kept,3] with volume anchors[3*i]; rows [n_kept, n_kept + n_edge) those at e_pts
 * [n_edge,3] with volume e_anc[i].  dparams_f32 (field MLP, 0 hidden matmuls) and grad_table [pool,2] are accumulated into;
 * dL/dinput is multiplied by grad_mul before it is scattered.  Same dL/dinput bits and per-run sums as the two-kernel sequence;
 * only the order of the fp32 reductions differs.  tcgen05 only. */
int f2b_field_bwd_scatter(const void* dout_f16, const void* in_f16, const void* params_f16, int n_kept, const float* pts,
                          const int* anchors, int n_edge, const float* e_pts, const int* e_anc, const int* prim_pool,
                          const float* bias_pool, int n_volumes, int local_size, float grad_mul, float* dparams_f32,
                          float* grad_table, void* stream);

/* Implementation selection for f2b_mlp_fwd / f2b_mlp_bwd: 1 = tcgen05/TMEM kernels (default when
 * built), 0 = CUDA-core twin (validation).  Env F2B_MLP_IMPL overrides the default. */
int f2b_set_mlp_impl(int impl);
int f2b_get_mlp_impl(void);
int f2b_mlp_fwd_v0(const void* in_f16, const void* params_f16, int n_hidden_matmuls, int n_pts,
                   void* out_f16, void* hidden_save_f16, void* stream);
int f2b_mlp_bwd_v0(const void* dout_f16, const void* in_f16, const void* hidden_save_f16,
                   const void* params_f16, int n_hidden_matmuls, int n_pts,
                   void* din_f16, float* dparams_f32, void* stream);
int f2b_mlp_fwd_tc(const void* in_f16, const void* params_f16, int n_hidden_matmuls, int n_pts,
                   void* out_f16, void* hidden_save_f16, void* stream);
int f2b_mlp_bwd_tc(const void* dout_f16, const void* in_f16, const void* hidden_save_f16,
                   const void* params_f16, int n_hidden_matmuls, int n_pts,
                   void* din_f16, float* dparams_f32, void* stream);

/* ------------------------------------------------------------------------------------------
 * Shader — replaces SHShader::Query (src/Shader/SHShader.cpp:23-29, SHShader.cu:10-118).
 * ------------------------------------------------------------------------------------------ */
int f2b_sh_encode(const float* dirs, int n_pts, int degree /* 1..4 */, float* out, void* stream);
/* CustomOps::ScatterIdx (Scatter.cu:110-131): per-ray camera index broadcast to the ray's samples. */
int f2b_scatter_idx(const int* pts_idx_bounds, const int* emb_idx, int n_rays, int* out, void* stream);
/* Shader-MLP input assembly (Renderer.cpp:179-187 + SHShader.cpp:24-25 + tcnn identity cast):
 * mlp_in[p] = fp16([1, scene_feat[p,1:16]] + app_emb[pt_emb_idx[p]] | SH4(dirs[p])); app_emb nullable. */
int f2b_shader_prep(const float* scene_feat /* [P,16] */, const float* dirs /* [P,3] */,
                    const float* app_emb /* [n_img,16] or NULL */, const int* pt_emb_idx /* [P] or NULL */,
                    int n_pts, void* mlp_in_f16 /* [P,32] */, void* stream);
/* rgb = (1+2e-3)*sigmoid(raw[:, :3]) - 1e-3 on the fp16 MLP output (SHShader.cpp:27-28). */
int f2b_shader_act(const void* raw_out_f16 /* [P,16] */, int n_pts, float* rgb /* [P,3] */, void* stream);
/* Backward of the activation: d_raw[P,16] fp16 = loss_scale * d_rgb * sigmoid' (channels 3..15 zero). */
int f2b_shader_act_bwd(const void* raw_out_f16, const float* d_rgb, int n_pts, float loss_scale,
                       void* d_raw_f16, void* stream);
/* Backward of the input assembly (one warp per ray): d_scene_feat[p,1:16] = d_mlp_in[p,1:16]*inv_loss_scale
 * (column 0 is left to the composite backward) and, when d_app_emb != NULL,
 * d_app_emb[emb_idx[ray]] += sum over the ray's samples of d_mlp_in[p,0:16]*inv_loss_scale
 * (ScatterAddFuncBackwardBlock, Scatter.cu:23-40). */
int f2b_shader_prep_bwd(const void* d_mlp_in_f16 /* [P,32] */, const int* pts_idx_bounds /* [R,2] */,
                        const int* emb_idx /* [R] or NULL */, int n_rays, float inv_loss_scale,
                        float* d_scene_feat /* [P,16] */, float* d_app_emb /* [n_emb,16] or NULL */, void* stream);
/* Same, fused with what follows it in the reference's graph: the slice/cat backward that puts the composite's
 * d logit into column 0 (Renderer.cpp:179-183) and TCNNWPFunction::backward's input scaling
 * (grad * loss_scale).to(fp16) (TCNNWP.cpp:213-216).  Emits the field MLP's dL/dout directly:
 * d_field_out[p,0] = half(d_logit[p]*field_loss_scale), d_field_out[p,k] = half(d_mlp_in[p,k]*inv_loss_scale*field_loss_scale). */
int f2b_shader_prep_bwd_f16(const void* d_mlp_in_f16 /* [P,32] */, const float* d_logit /* [P] */,
                            const int* pts_idx_bounds, const int* emb_idx, int n_rays, float inv_loss_scale,
                            float field_loss_scale, void* d_field_out_f16 /* [P,16] */, float* d_app_emb, void* stream);

/* ------------------------------------------------------------------------------------------
 * Octree maintenance on the device (SURVEY §8f N2) — replaces PersOctree::ProcOctree(compact = true, subdivide,
 * brute_force) (src/PtsSampler/PersSampler.cpp:120-330: prune dead leaves, collapse single-child chains, renumber,
 * optionally split every leaf visited more than 4 times into 8; called from PersSampler::UpdateOctNodes,
 * PersSampler.cu:604-614) and PersOctree::MarkInvisibleNodes (PersSampler.cu:616-680).  Same node numbering, links,
 * centres and statistics as the reference's sequential host pass, without the three D2H + three H2D blob copies.
 * work_nodes: [n_nodes] TreeNode scratch; work_i32: [5*n_nodes + 2] ints; outputs sized for 9*n_nodes nodes;
 * n_nodes_out: device int (the only value the host has to read back); visit counts restart at zero (caller memsets).
 * ------------------------------------------------------------------------------------------ */
int f2b_octree_proc(const void* tree_nodes, const int* weight_stats, const int* alpha_stats, const int* visit_cnt,
                    int n_nodes, int subdivide, int brute_force, void* work_nodes, int* work_i32, void* nodes_out,
                    int* weight_stats_out, int* alpha_stats_out, int* n_nodes_out, void* stream);
/* nodes no training camera can see get trans_idx = -1.  intri [n_cams,3,3], w2c [n_cams,3,4], bounds [n_cams,2]. */
int f2b_octree_mark_invisible(void* tree_nodes, int n_nodes, const float* intri, const float* w2c, const float* bounds,
                              int n_cams, void* stream);

/* ------------------------------------------------------------------------------------------
 * Ray generation (SURVEY §8f N3) — replaces Dataset::Img2WorldRayFlex / Img2WorldRayKernel incl. the Newton
 * undistortion (src/Dataset/Dataset.cu:30-74,100-152) and the CPU ground-truth gather + H2D copy of
 * Dataset::RandRaysData (src/Dataset/Dataset.cpp:290).  poses [n_cam,3,4], intri [n_cam,3,3], dist_params [n_cam,4]
 * (k1,k2,p1,p2) fp32 row-major as Dataset holds them; cam_indices [n] i32; ij [n,2] i32 = (row, col), the +0.5 pixel
 * centre is applied inside.  Bit-identical rays (operation order from the reference's PTX).
 * ------------------------------------------------------------------------------------------ */
int f2b_img2world_rays(const float* poses, const float* intri, const float* dist_params, const int* cam_indices,
                       const int* ij, int n_rays, float* rays_o /* [n,3] */, float* rays_d /* [n,3], not normalised */,
                       void* stream);
/* out[r] = images[cam_indices[r], ij[r,0], ij[r,1], 0:3]; images fp32 [n_img, height, width, 3] resident on the device. */
int f2b_gather_pixels(const float* images, const int* cam_indices, const int* ij, int height, int width, int n,
                      float* out /* [n,3] */, void* stream);

/* ------------------------------------------------------------------------------------------
 * Optimizer step (SURVEY §8f N1) — replaces torch::optim::Adam::step for one parameter tensor
 * (built at src/ExpRunner.cpp:54 from Hash3DAnchored::OptimParamGroups, src/Field/Hash3DAnchored.cpp:124-150;
 * stepped at ExpRunner.cpp:136) and, when shadow_f16 != NULL, the fp32->fp16 table copy of the next forward
 * (Hash3DAnchored.cu:186).  Same arithmetic, order and roundings as the ATen elementwise sequence, in one pass.
 * Only elements [0, n_live) are read/written (n_live % 4 == 0): pass the live prefix of the hash table
 * (17/32 of the pool), n for the other parameters.  step = 1 for the first update.
 * ------------------------------------------------------------------------------------------ */
int f2b_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, int64_t n_live,
                  double lr, double beta1, double beta2, double eps, double weight_decay, int64_t step,
                  void* shadow_f16 /* [n] fp16 or NULL */, void* stream);

/* ------------------------------------------------------------------------------------------
 * Composite — replaces the Renderer::Render tail (src/Renderer/Renderer.cpp:107-150,196-208),
 * FlexOps::{Sum,AccumulateSum} (src/Utils/CustomOps/FlexOps.cu), TruncExp (CustomOps.cpp:9-18),
 * FilterIdxBounds/CountValidPts (Renderer.cu:8-50) and the gather-compaction (Renderer.cpp:126-132).
 * All per-ray sums run in the reference's serial left-to-right order (bit-compatible rounding).
 * ------------------------------------------------------------------------------------------ */
/* No-grad early-stop pass: density logit (scene_feat[:,0], element stride logit_stride) + dt ->
 * weights, alphas (for UpdateOctNodes), keep mask (trans > 1e-4) and the compacted bounds. */
int f2b_early_stop(const float* logit, int logit_stride, const float* dt, const int* pts_idx_bounds,
                   int n_rays, float* weights, float* alphas, uint8_t* keep,
                   int* ray_counts /* [n_rays] caller-owned scratch */,
                   int* new_bounds /* [n_rays,2] */, int* total_kept /* [1] */, void* stream);
/* The two halves of f2b_early_stop separately (ray-chunked pipelines scan once over all chunks' counts). */
int f2b_early_stop_rays(const float* logit, int logit_stride, const float* dt, const int* pts_idx_bounds,
                        int n_rays, float* weights, float* alphas, uint8_t* keep, int* ray_counts, void* stream);
/* counts[n] -> bounds[n,2] = {exclusive, inclusive} prefix sums, total[0] = sum (torch::cumsum at
 * PersSampler.cu:395 / FilterIdxBounds, Renderer.cu:8-29). */
int f2b_count_scan(const int* counts, int n, int* bounds, int* total, void* stream);
/* slot_bounds[r] = {(first_ray+r)*slot_size, (first_ray+r)*slot_size + ray_counts[r]}: pts_idx_bounds of the scratch layout. */
int f2b_slot_bounds(const int* ray_counts, int n_rays, int slot_size, int first_ray, int* slot_bounds, void* stream);
/* f2b_compact_samples reading the march's scratch slots directly (28 B/sample there: pts, dt, t, anchors[0:2]); the
 * per-sample direction is the ray's (rays_d [n_rays,3], normalised), anchors_o[:,2] = 0. */
int f2b_compact_slots(const uint8_t* keep, const int* slot_bounds, const int* new_bounds, int n_rays,
                      const float* rays_d, const float* s_pts, const float* s_dt, const float* s_t,
                      const int* s_anchors, const void* feat_slots_f16 /* nullable */, float* pts_o, float* dirs_o,
                      float* dt_o, float* t_o, int* anchors_o, void* feat_o_f16 /* nullable */, void* stream);
/* Gather-compact the surviving samples (44 B/pt) and, optionally, their encoded features (feat_f16 [P,32]
 * from the early-stop pass -> feat_o_f16 [P',32]) so the gradient pass does not gather the table again. */
int f2b_compact_samples(const uint8_t* keep, const int* old_bounds, const int* new_bounds, int n_rays,
                        const float* pts, const float* dirs, const float* dt, const float* t,
                        const int* anchors, const void* feat_f16 /* nullable */,
                        float* pts_o, float* dirs_o, float* dt_o, float* t_o, int* anchors_o,
                        void* feat_o_f16 /* nullable */, void* stream);
/* Forward composite. logit: scene_feat[:,0] (stride logit_stride); rgb [P,3]; t is the raw sample t
 * (the +1e-2 of Renderer.cpp:197 is applied inside).  Outputs per ray: colors[3], disparity, depth;
 * per point: weights. */
int f2b_composite_fwd(const float* logit, int logit_stride, const float* rgb, const float* dt,
                      const float* t, const int* pts_idx_bounds, const float* bg_color, int n_rays,
                      float* colors, float* disparity, float* depth, float* weights, void* stream);
/* Backward of the above (+ TruncExp backward + optional GradientScaling, CustomOps.cu:68-80):
 * given dL/dcolors [R,3], dL/ddisparity [R], dL/ddepth [R] (nullable), dL/dweights [P] (nullable)
 * -> dL/dlogit [P] (written with stride dlogit_stride), dL/drgb [P,3].
 * grad_scaling_progress >= 1 disables gradient scaling. */
int f2b_composite_bwd(const float* logit, int logit_stride, const float* rgb, const float* dt,
                      const float* t, const int* pts_idx_bounds, const float* bg_color, int n_rays,
                      const float* d_colors, const float* d_disparity, const float* d_depth,
                      const float* d_weights, float grad_scaling_progress,
                      float* d_logit, int dlogit_stride, float* d_rgb, void* stream);
/* f2b_composite_bwd with the colour activation's backward (f2b_shader_act_bwd) applied on the way out: instead of
 * d_rgb [P,3] fp32 it writes the shader MLP's dL/dout row d_raw [P,16] fp16 = loss_scale * d_rgb * sigmoid'(raw), 0 x 13. */
int f2b_composite_act_bwd(const float* logit, int logit_stride, const float* rgb, const float* dt, const float* t,
                          const int* pts_idx_bounds, const float* bg_color, int n_rays, const float* d_colors,
                          const float* d_disparity, const float* d_depth, const float* d_weights,
                          float grad_scaling_progress, const void* raw_f16 /* [P,16] */, float loss_scale,
                          float* d_logit, int dlogit_stride, void* d_raw_f16 /* [P,16] */, void* stream);
/* Stand-alone FlexOps (FlexOps.h:15-16) for callers that use them directly. */
int f2b_flex_sum(const float* val, int vec, const int* idx_start_end, int n_outs, float* sum, void* stream);
int f2b_flex_accumulate_sum(const float* val, const int* idx_start_end, int n_outs, int include_this,
                            float* out, void* stream);
/* WeightVar loss forward/backward (CustomOps.cu:12-66). */
int f2b_weight_var_fwd(const float* weights, const int* idx_start_end, int n_outs, float* out_vars, void* stream);
int f2b_weight_var_bwd(const float* weights, const int* idx_start_end, int n_outs, const float* dl_dvars,
                       float* dl_dw, void* stream);

/* ------------------------------------------------------------------------------------------
 * Renderer::Render (src/Renderer/Renderer.cpp:52-213) as THREE launch sequences — what the host mirrors call per batch.
 * Each entry point enqueues the fixed kernel sequence of one phase of the fused pipeline (the very kernels declared above,
 * same order, same streams) in ONE call, so that a scripting-language host pays one foreign call per phase instead of one
 * per kernel; nothing is allocated, every buffer (and the two streams) comes from the caller in `f2b_render`.  Fields a
 * phase does not use may be left NULL / 0.  The host keeps what only it can do: the torch RNG draws (noise, background,
 * edge indices / coordinates), the ONE host sync between phase 1 and phase 2 (n_kept sizes the survivors' buffers),
 * the GlobalDataPool EMAs and the autograd plumbing.
 *   f2b_render_phase1      [march + slot bounds unless skip_march] -> field-parameter cast -> early-stop field pass on the
 *                          slots -> per-ray early stop -> survivor count scan                    (Renderer.cpp:52-126)
 *   f2b_render_phase2_fwd  compaction -> [TRAIN: edge points + their encode] -> point->camera index -> parameter casts ->
 *                          field MLP + shader-input epilogue -> edge-point MLP -> shader MLP + colour activation ->
 *                          composite                                                             (Renderer.cpp:127-208)
 *   f2b_render_bwd         zero-fills -> composite/activation bwd -> shader MLP bwd -> input-assembly bwd -> scatter_mode 0:
 *                          field MLP bwd + hash scatter of ray samples and edge points in one kernel (f2b_field_bwd_scatter;
 *                          F2B_FIELD_BWD_SCATTER=0: field MLP bwd into dfeat16, the scatter of both on side_stream, joined);
 *                          scatter_mode 1: field MLP bwd into dfeat16 only (the caller scatters it by level slabs)
 *   f2b_render_grad_finalize  un-scale the two MLP gradients (TCNNWP.cpp:225-229) and raise the per-MLP non-finite flags
 *                          (dL/dparams, and dL/dinput through d_app / the live table gradient; TCNNWP.cpp:231-240)
 * ------------------------------------------------------------------------------------------ */
typedef struct f2b_render {
  /* scene blobs + sampler settings (PersSampler) */
  const void* tree_nodes; int n_nodes; const void* trans; int n_trans; const void* edge_pool;
  float near_t, far_t, sample_l; int scale_by_dis, max_hits, count_all_hits;
  /* field / shader parameters: fp32 masters, fp16 copies written by phase1 (field) and phase2_fwd (both) */
  const void* table16; const int* prim; const float* bias; int n_volumes, local_size;
  const float* field_params; int n_field_params; const float* shader_params; int n_shader_params;
  void* fparams16; void* sparams16;
  const float* app_emb; int n_emb;                       /* NULL: no appearance embedding */
  /* the ray batch */
  int n_rays; const float* rays_o; const float* rays_d /* normalised */; const float* noise; const float* bg;
  const int* ray_emb_idx;                                /* [n_rays] or NULL */
  /* phase 1: slot layout (ray r owns slots [r*1024, r*1024 + counts[r])) */
  int skip_march;                                        /* 1: the slots were marched ahead of time (prefetch) */
  float* s_pts; float* s_dt; float* s_t; int* s_anchors; int* counts; int* chunk_bounds; int* slot_bounds;
  float* first_oct_dis; int* totals /* [2] */;
  float* logit_s; void* feat_s; float* w0; float* a0; uint8_t* keep; int* kept_counts; int* new_bounds; int* total_kept;
  /* phase 2: survivors (n_kept rows) + TV-loss edge points (2 * n_edge_pairs rows behind them in feat_q / f_hidden / dfeat16) */
  int n_kept; int n_edge_pairs;
  float* pts; float* dirs; float* dt; float* t; int* anchors; void* feat_q;
  const int* edge_idx; const float* edge_coord; float* e_pts; int* e_anc;
  int* pt_emb_idx;                                       /* [n_kept] scratch, used when app_emb && ray_emb_idx */
  float* logit; void* mlp_in; void* f_hidden /* nullable */; float* edge32; void* raw; float* rgb; void* s_hidden /* nullable */;
  float* colors; float* disparity; float* depth; float* weights;
  /* backward */
  const float* d_colors; const float* d_disparity; const float* d_depth; const float* d_weights; const float* d_edge /* [2*pairs,16] */;
  float gs_progress, shader_loss_scale, field_loss_scale, table_grad_mul;
  float* d_logit; void* d_raw; void* d_in16; void* d_scene16; void* dfeat16 /* unused (may be NULL) by the one-kernel scatter */;
  float* d_sparams; float* d_fparams; float* d_table; int64_t table_numel; int64_t table_live; float* d_app;
  int scatter_mode;                                      /* 0: scatter inside f2b_render_bwd; 1: the caller scatters (level slabs) */
  int* nonfinite;                                        /* [2] device ints: shader MLP, field MLP */
  void* stream; void* side_stream;
} f2b_render;
int f2b_render_sizeof(void);                 /* sizeof(f2b_render) as the library was built: bindings compare it with their own */
int f2b_render_phase1(const f2b_render* r);
int f2b_render_phase2_fwd(const f2b_render* r);
int f2b_render_bwd(const f2b_render* r);
int f2b_render_grad_finalize(const f2b_render* r);

/* ---- forward-only (VALIDATE / no-grad) Renderer::Render behind the march as ONE kernel --------------------------------
 * Replaces Renderer.cpp:107-208 for a batch that takes no gradient (ExpRunner::RenderWholeImage, ExpRunner.cpp:257-293):
 * hash encode -> field MLP -> early stop (T > 1e-4, Renderer.cpp:125) -> shading-feature assembly + SH4 -> shader MLP ->
 * colour activation -> composite, one CTA walking one ray front to back over the march's slot layout
 * (slot_pts [R*slot,3], slot_dt / slot_t [R*slot], slot_anchors [R*slot,2], ray_counts [R] as f2b_sampler_march leaves them)
 * and stopping at the first opaque sample — the samples behind it are never encoded.  No app embedding (Renderer.cpp:184
 * applies it in TRAIN mode only).  rays_d normalised, bg [R,3].  total_all: device int, the batch's sample total (NULL or
 * > 0: normal; <= 0: the reference's empty-batch result, depth = 512, Renderer.cpp:83-97).  ticket: [1] device int scratch.
 * Outputs: colors [R,3], disparity [R], depth [R], kept_counts [R] (survivors per ray), and — nullable — weights_slots
 * [R*slot]: the kept samples' weights at their slots (f2b_gather_kept_weights packs them into RenderResult.weights order).
 * Values are bit-identical to f2b_render_phase1 + f2b_render_phase2_fwd on the same batch.  tcgen05 implementation only. */
int f2b_render_fwd_fused(const void* table_f16, const int* prim_pool, const float* bias_pool, int n_volumes, int local_size,
                         const void* field_params_f16, const void* shader_params_f16, const float* slot_pts, const float* slot_dt,
                         const float* slot_t, const int* slot_anchors, const int* ray_counts, const float* rays_d, const float* bg,
                         int n_rays, int slot_size, const int* total_all, int* ticket, float* colors, float* disparity,
                         float* depth, int* kept_counts, float* weights_slots, void* stream);
/* weights_slots [R*slot] + new_bounds [R,2] (f2b_count_scan of kept_counts) -> weights [P'] in the packed ray order. */
int f2b_gather_kept_weights(const float* weights_slots, const int* new_bounds, int n_rays, int slot_size, float* weights,
                            void* stream);

#ifdef __cplusplus
}
#endif
#endif /* F2NERF_B200_H */
