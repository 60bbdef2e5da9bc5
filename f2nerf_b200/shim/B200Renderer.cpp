// B200Renderer.cpp — the fused C++/LibTorch host of the hot path: a replacement BODY for the reference's
// `RenderResult Renderer::Render(rays_o, rays_d, bounds, emb_idx)` (src/Renderer/Renderer.cpp:52-213).
//
// The reference's Renderer CLASS is kept as it is (constructor, factories, States/LoadStates, OptimParamGroups,
// app_emb_, the PersSampler / Hash3DAnchored / SHShader objects it builds): this file only supplies the member
// function `Renderer::Render`, so an unmodified ExpRunner (src/ExpRunner.cpp:65-186: RandRaysData -> Render -> loss ->
// backward -> Adam) trains through the B200 kernels.  How the body is swapped without touching a reference source
// line is a build-recipe matter (INTEGRATION.md section 3): the reference's Renderer.cpp is compiled with
// -DRender=RenderReference (its own body stays callable under that name, see RenderReferenceThunk.cpp), this file
// is compiled without the macro.  Setting F2B_RENDER=reference at run time routes every call back to the reference body.
//
// Same pipeline as the Python host mirror (f2nerf_b200/renderer.py), kernel for kernel, through the flat C ABI
// (include/f2nerf_b200.h): one-pass march into per-ray slots -> early-stop field pass on the slots -> per-ray
// survivor counts -> ONE host sync -> compaction (samples + their encoded features) -> fused field-MLP / shader-input
// epilogue -> shader MLP + colour activation -> composite; ONE autograd node carries the whole backward
// (composite+activation bwd -> shader MLP bwd -> input-assembly bwd -> field MLP bwd -> hash scatter).
// RNG: the same torch draws in the same order as the reference (noise, background, edge samples) and the Philox
// offset advanced by what the reference's torch::rand MLP-output buffers (TCNNWP.cpp:143) and GradientScaling's
// rand_like (CustomOps.cu:154) would have consumed, so a seeded run stays on the reference's random stream.
#include <torch/torch.h>
#include <ATen/cuda/CUDAContext.h>
#include <ATen/cuda/CUDAGeneratorImpl.h>
#include <ATen/cuda/CUDAEvent.h>
#include <c10/cuda/CUDAStream.h>
#include <c10/cuda/CUDAGuard.h>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <mutex>
#include <unordered_map>
#include "Common.h"
#include "Renderer/Renderer.h"
#include "PtsSampler/PersSampler.h"
#include "Field/Hash3DAnchored.h"
#include "Shader/SHShader.h"
#include "f2nerf_b200.h"
#include "B200Renderer.h"

using Tensor = torch::Tensor;
using torch::autograd::AutogradContext;
using torch::autograd::variable_list;

RenderResult f2b_reference_render(Renderer* r, const Tensor& rays_o, const Tensor& rays_d, const Tensor& bounds,
                                  const Tensor& emb_idx);                    // RenderReferenceThunk.cpp

#define F2B_CHECK(expr)                                                            \
  do {                                                                             \
    int f2b_rc_ = (expr);                                                          \
    CHECK(f2b_rc_ == 0) << #expr << " -> " << f2b_rc_ << ": " << f2b_last_error(); \
  } while (0)

static bool g_keep_samples = [] { const char* e = std::getenv("F2B_KEEP_SAMPLES"); return e && e[0] == '1'; }();
static bool g_use_reference = [] { const char* e = std::getenv("F2B_RENDER"); return e && std::string(e) == "reference"; }();
void f2b_render_keep_samples(bool on) { g_keep_samples = on; }
void f2b_render_use_reference(bool on) { g_use_reference = on; }

namespace {

constexpr int kSlot = 1024;            // MAX_SAMPLE_PER_RAY (PersSampler.h:9)
constexpr int kEdgePts = 8192;         // Renderer.cpp:155
const auto kHalf = torch::TensorOptions().dtype(torch::kFloat16).device(torch::kCUDA);
const auto kByte = torch::TensorOptions().dtype(torch::kUInt8).device(torch::kCUDA);

void* cur_stream() { return (void*) at::cuda::getCurrentCUDAStream().stream(); }
void* P(const Tensor& t) { return t.defined() ? t.data_ptr() : nullptr; }
// F2B_MLP_RECOMPUTE (default 1): the MLP forward saves no hidden activations, f2b_mlp_bwd2(hidden0 = NULL) rebuilds them
// F2B_FUSED_FORWARD (default 1): VALIDATE-mode Render = march + f2b_render_fwd_fused; F2B_VALIDATE_WEIGHTS (default 1): also pack
// RenderResult.weights / idx_start_end (costs the step's one host read)
bool fused_forward() {
  static const bool on = [] { const char* e = getenv("F2B_FUSED_FORWARD"); return !e || atoi(e) != 0; }();
  return on;
}
// F2B_FIELD_BWD_SCATTER (default 1): the field-MLP backward and the hash scatter as one kernel (f2b_field_bwd_scatter); 0 runs
// f2b_mlp_bwd2 -> dfeat16 -> f2b_hash_bwd (the same switch as the Python host's)
bool field_bwd_scatter() {
  static const bool on = [] { const char* e = getenv("F2B_FIELD_BWD_SCATTER"); return !e || atoi(e) != 0; }();
  return on;
}
bool validate_weights() {
  static const bool on = [] { const char* e = getenv("F2B_VALIDATE_WEIGHTS"); return !e || atoi(e) != 0; }();
  return on;
}
// F2B_SHIM_PROFILE=1: host wall time spent inside Render (TRAIN / VALIDATE) and inside its backward, printed at exit — what share of
// a trainer iteration the path is (both contain the waits for their own GPU work: Render ends behind the survivor-count read, the
// backward behind its NaN-flag read)
struct ShimProfile {
  bool on = false;
  double t_render_train = 0, t_render_val = 0, t_backward = 0;
  long n_train = 0, n_val = 0, n_bwd = 0;
  ShimProfile() { const char* e = getenv("F2B_SHIM_PROFILE"); on = e && atoi(e) != 0; }
  ~ShimProfile() {
    if (on)
      std::printf("{\"f2b_shim_profile\": {\"render_train_s\": %.3f, \"n_render_train\": %ld, \"render_validate_s\": %.3f, "
                  "\"n_render_validate\": %ld, \"backward_s\": %.3f, \"n_backward\": %ld}}\n",
                  t_render_train, n_train, t_render_val, n_val, t_backward, n_bwd);
  }
};
ShimProfile g_prof;
struct ScopedTimer {
  double* acc; long* cnt; std::chrono::steady_clock::time_point t0;
  ScopedTimer(double* a, long* c) : acc(g_prof.on ? a : nullptr), cnt(c), t0(std::chrono::steady_clock::now()) {}
  ~ScopedTimer() { if (acc) { *acc += std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count(); ++*cnt; } }
};

bool mlp_recompute() {
  static const bool on = [] { const char* e = getenv("F2B_MLP_RECOMPUTE"); return !e || atoi(e) != 0; }();
  return on;
}
float* PF(const Tensor& t) { return t.defined() ? t.data_ptr<float>() : nullptr; }
int* PI(const Tensor& t) { return t.defined() ? t.data_ptr<int>() : nullptr; }

// ---- RNG-stream parity (see f2nerf_b200/rng.py): advance the Philox offset as ATen's uniform kernel would ---------
void burn_rand(int64_t numel) {
  if (numel <= 0) return;
  const auto* prop = at::cuda::getCurrentDeviceProperties();
  const int64_t block = 256, unroll = 4;
  const int64_t max_grid = int64_t(prop->multiProcessorCount) * (prop->maxThreadsPerMultiProcessor / block);
  const int64_t grid = std::min(max_grid, (numel + block - 1) / block);
  const uint64_t inc = uint64_t(((numel - 1) / (block * grid * unroll) + 1) * 4);
  auto gen = at::cuda::detail::getDefaultCUDAGenerator();
  auto* impl = at::check_generator<at::CUDAGeneratorImpl>(gen);
  std::lock_guard<std::mutex> lock(impl->mutex_);
  impl->set_philox_offset_per_thread(impl->philox_offset_per_thread() + inc);
}
void burn_mlp_output(int64_t batch) { if (batch > 0) burn_rand(((batch + 127) / 128 * 128) * 16); }

// ---- persistent per-renderer work buffers (slot layout; grown on demand, no allocator traffic in steady state) ----
struct Work {
  int64_t cap_rays = 0;
  Tensor s_pts, s_dt, s_t, s_anchors, logit_s, feat_s, w0, a0, keep, kept_counts, table16;
  c10::Storage d_table_storage;          // the table gradient's storage, kept across steps (its dead 15/32 stays zero)
  c10::optional<c10::cuda::CUDAStream> side_votes, side_scatter;
  void ensure(int64_t n_rays, int64_t table_numel) {
    if (n_rays > cap_rays) {
      const int64_t n = n_rays * kSlot;
      s_pts = torch::empty({n, 3}, CUDAFloat); s_dt = torch::empty({n}, CUDAFloat); s_t = torch::empty({n}, CUDAFloat);
      s_anchors = torch::empty({n, 2}, CUDAInt);
      logit_s = torch::empty({n}, CUDAFloat); feat_s = torch::empty({n, 32}, kHalf);
      w0 = torch::empty({n}, CUDAFloat); a0 = torch::empty({n}, CUDAFloat); keep = torch::empty({n}, kByte);
      kept_counts = torch::empty({n_rays}, CUDAInt);
      cap_rays = n_rays;
    }
    if (!table16.defined() || table16.numel() != table_numel) table16 = torch::empty({table_numel}, kHalf);
    if (!side_votes) { side_votes = c10::cuda::getStreamFromPool(); side_scatter = c10::cuda::getStreamFromPool(); }
  }
};
Work& work_of(const Renderer* r) {
  static std::unordered_map<const Renderer*, Work> pool;
  return pool[r];
}

void stream_wait(const c10::cuda::CUDAStream& waiter, const c10::cuda::CUDAStream& on) {
  at::cuda::CUDAEvent ev;
  ev.record(on);
  ev.block(waiter);
}

// What the second half of Render hands to its autograd node (plain struct; lives in the node through a registry slot).
struct Pack {
  Renderer* renderer = nullptr;
  Hash3DAnchored* field = nullptr;
  SHShader* shader = nullptr;
  Tensor pts, dirs, dt, t, anchors, bounds, bg, feat16, e_pts, e_anc, pt_emb_idx, ray_emb_idx;
  int64_t n_kept = 0, n_edge = 0;
  bool grad_on = false;
  float gs_progress = 1.f;
  // saved by forward
  Tensor fparams16, sparams16, logit, mlp_in, raw, rgb, f_hidden, s_hidden;
};
std::mutex g_pack_mu;
std::unordered_map<int64_t, std::shared_ptr<Pack>> g_packs;
int64_t g_pack_next = 1;

class RenderFn : public torch::autograd::Function<RenderFn> {
public:
  static variable_list forward(AutogradContext* ctx, Tensor feat_pool, Tensor field_params, Tensor shader_params, Tensor app_emb,
                               int64_t pack_id) {
    std::shared_ptr<Pack> pk;
    { std::lock_guard<std::mutex> l(g_pack_mu); pk = g_packs.at(pack_id); }
    Pack& k = *pk;
    const int64_t n_kept = k.n_kept, n_q = k.feat16.size(0);
    k.fparams16 = torch::empty({field_params.numel()}, kHalf);
    k.sparams16 = torch::empty({shader_params.numel()}, kHalf);
    F2B_CHECK(f2b_cast_f32_to_f16(field_params.data_ptr<float>(), P(k.fparams16), field_params.numel(), 1.f, cur_stream()));
    F2B_CHECK(f2b_cast_f32_to_f16(shader_params.data_ptr<float>(), P(k.sparams16), shader_params.numel(), 1.f, cur_stream()));
    const bool emb_on = k.pt_emb_idx.defined();
    const bool save = k.grad_on && !mlp_recompute();
    if (save) k.f_hidden = torch::empty({1, n_q, 64}, kHalf);
    k.logit = torch::empty({n_kept}, CUDAFloat);
    k.mlp_in = torch::empty({n_kept, 32}, kHalf);
    F2B_CHECK(f2b_field_shade_fwd(P(k.feat16), P(k.fparams16), PF(k.dirs), emb_on ? app_emb.data_ptr<float>() : nullptr,
                                  emb_on ? PI(k.pt_emb_idx) : nullptr, (int) n_kept, PF(k.logit), P(k.mlp_in),
                                  P(k.f_hidden), cur_stream()));
    Tensor edge32 = torch::empty({n_q - n_kept, 16}, CUDAFloat);
    if (n_q > n_kept) {
      F2B_CHECK(f2b_mlp_fwd_f32((char*) P(k.feat16) + n_kept * 64, P(k.fparams16), 0, (int) (n_q - n_kept), PF(edge32), nullptr,
                                save ? (void*) ((char*) P(k.f_hidden) + n_kept * 128) : nullptr, cur_stream()));
    }
    if (save) k.s_hidden = torch::empty({2, n_kept, 64}, kHalf);
    k.raw = torch::empty({n_kept, 16}, kHalf);
    k.rgb = torch::empty({n_kept, 3}, CUDAFloat);
    F2B_CHECK(f2b_shader_mlp_rgb_fwd(P(k.mlp_in), P(k.sparams16), (int) n_kept, P(k.raw), PF(k.rgb),
                                     P(k.s_hidden), cur_stream()));
    const int n_rays = k.bounds.size(0);
    Tensor colors = torch::empty({n_rays, 3}, CUDAFloat), disp = torch::empty({n_rays}, CUDAFloat),
           depth = torch::empty({n_rays}, CUDAFloat), weights = torch::empty({n_kept}, CUDAFloat);
    F2B_CHECK(f2b_composite_fwd(PF(k.logit), 1, PF(k.rgb), PF(k.dt), PF(k.t), PI(k.bounds), PF(k.bg), n_rays, PF(colors),
                                PF(disp), PF(depth), PF(weights), cur_stream()));
    ctx->saved_data["pack"] = pack_id;
    ctx->saved_data["table_numel"] = feat_pool.numel();
    ctx->saved_data["n_emb"] = app_emb.size(0);
    return {colors, disp, depth, weights, edge32.reshape({-1, 2, 16})};
  }

  static variable_list backward(AutogradContext* ctx, variable_list g) {
    ScopedTimer prof_timer(&g_prof.t_backward, &g_prof.n_bwd);
    const int64_t pack_id = ctx->saved_data["pack"].toInt();
    std::shared_ptr<Pack> pk;
    {
      std::lock_guard<std::mutex> l(g_pack_mu);
      auto it = g_packs.find(pack_id);
      CHECK(it != g_packs.end()) << "Renderer::Render backward: the saved activations were released by a previous backward";
      pk = it->second;
      g_packs.erase(it);                         // like tiny-cuda-nn's context (TCNNWP.cpp:207) the graph is traversed once
    }
    Pack& k = *pk;
    CHECK(k.grad_on) << "Renderer::Render backward: forward ran without grad (VALIDATE mode / NoGradGuard)";
    const int64_t n_kept = k.n_kept, n_q = k.feat16.size(0);
    const int n_rays = k.bounds.size(0);
    Hash3DAnchored* field = k.field;
    SHShader* shader = k.shader;
    Tensor d_colors = g[0].defined() ? g[0].contiguous() : torch::zeros({n_rays, 3}, CUDAFloat);
    Tensor d_disp = g[1].defined() ? g[1].contiguous() : Tensor();
    Tensor d_depth = g[2].defined() ? g[2].contiguous() : Tensor();
    Tensor d_weights = g[3].defined() ? g[3].contiguous() : Tensor();
    Tensor d_edge = g[4];
    if (k.gs_progress < 1.f) { burn_rand(n_kept * 3); burn_rand(n_kept); }       // GradientScaling::backward's rand_like
    const float s_scale = shader->mlp_->loss_scale_, f_scale = field->mlp_->loss_scale_;
    Tensor d_logit = torch::empty({n_kept}, CUDAFloat);
    Tensor d_raw = torch::empty({n_kept, 16}, kHalf), d_in16 = torch::empty({n_kept, 32}, kHalf);
    Tensor d_scene16 = torch::empty({n_q, 16}, kHalf);
    Tensor d_sparams = torch::zeros({k.sparams16.numel()}, CUDAFloat), d_fparams = torch::zeros({k.fparams16.numel()}, CUDAFloat);
    const int64_t table_numel = ctx->saved_data["table_numel"].toInt();
    const int local_size = ((field->pool_size_ / N_LEVELS) >> 4) << 4;
    const int64_t live = std::min<int64_t>(table_numel, int64_t(N_LEVELS + 1) * local_size);     // halves [0, 17 S) are ever addressed
    // Only floats [0, 17 S) of the gradient are ever written, so its storage is kept across steps and only that live prefix is
    // zero-filled per backward — unless a tensor on last step's gradient is still alive (a trainer that keeps .grad): then a fresh,
    // fully zeroed one.  Each backward hands autograd a NEW tensor on the storage, so it becomes .grad without a copy.
    Work& wk = work_of(k.renderer);
    Tensor d_table;
    if (wk.d_table_storage && wk.d_table_storage.nbytes() == size_t(table_numel) * 4 && wk.d_table_storage.use_count() == 1) {
      d_table = torch::empty({0}, CUDAFloat).set_(wk.d_table_storage, 0, {table_numel / 2, 2});
      d_table.view({-1}).slice(0, 0, live).zero_();
    } else {
      d_table = torch::zeros({table_numel / 2, 2}, CUDAFloat);
      wk.d_table_storage = d_table.storage();
    }
    const bool emb_on = k.ray_emb_idx.defined();
    Tensor d_app = emb_on ? torch::zeros({ctx->saved_data["n_emb"].toInt(), 16}, CUDAFloat) : Tensor();
    if (n_q > n_kept) {
      if (d_edge.defined()) d_scene16.slice(0, n_kept, n_q).copy_((d_edge.reshape({-1, 16}) * f_scale).to(torch::kFloat16));
      else d_scene16.slice(0, n_kept, n_q).zero_();
    }
    F2B_CHECK(f2b_composite_act_bwd(PF(k.logit), 1, PF(k.rgb), PF(k.dt), PF(k.t), PI(k.bounds), PF(k.bg), n_rays, PF(d_colors),
                                    PF(d_disp), PF(d_depth), PF(d_weights), k.gs_progress, P(k.raw), s_scale, PF(d_logit), 1,
                                    P(d_raw), cur_stream()));
    F2B_CHECK(f2b_mlp_bwd2(P(d_raw), P(k.mlp_in), P(k.s_hidden),
                           k.s_hidden.defined() ? (void*) ((char*) P(k.s_hidden) + n_kept * 128) : nullptr, P(k.sparams16), 1,
                           (int) n_kept, P(d_in16), PF(d_sparams), cur_stream()));
    F2B_CHECK(f2b_shader_prep_bwd_f16(P(d_in16), PF(d_logit), PI(k.bounds), emb_on ? PI(k.ray_emb_idx) : nullptr, n_rays,
                                      1.f / s_scale, f_scale, P(d_scene16), PF(d_app), cur_stream()));
    if (field_bwd_scatter()) {
      F2B_CHECK(f2b_field_bwd_scatter(P(d_scene16), P(k.feat16), P(k.fparams16), (int) n_kept, PF(k.pts), PI(k.anchors),
                                      (int) (n_q - n_kept), n_q > n_kept ? PF(k.e_pts) : nullptr, n_q > n_kept ? PI(k.e_anc) : nullptr,
                                      field->prim_pool_.data_ptr<int>(), field->bias_pool_.data_ptr<float>(), field->n_volumes_,
                                      local_size, 1.f / f_scale, PF(d_fparams), PF(d_table), cur_stream()));
    } else {
      Tensor dfeat16 = torch::empty({n_q, 32}, kHalf);
      F2B_CHECK(f2b_mlp_bwd2(P(d_scene16), P(k.feat16), P(k.f_hidden), nullptr, P(k.fparams16), 0, (int) n_q, P(dfeat16),
                             PF(d_fparams), cur_stream()));
      F2B_CHECK(f2b_hash_bwd(field->prim_pool_.data_ptr<int>(), field->bias_pool_.data_ptr<float>(), field->n_volumes_, local_size,
                             PF(k.pts), PI(k.anchors), 3, (int) n_kept, P(dfeat16), 1, 1.f / f_scale, PF(d_table), cur_stream()));
      if (n_q > n_kept) {
        F2B_CHECK(f2b_hash_bwd(field->prim_pool_.data_ptr<int>(), field->bias_pool_.data_ptr<float>(), field->n_volumes_, local_size,
                               PF(k.e_pts), PI(k.e_anc), 1, (int) (n_q - n_kept), (char*) P(dfeat16) + n_kept * 64, 1, 1.f / f_scale,
                               PF(d_table), cur_stream()));
      }
    }
    d_sparams = d_sparams / s_scale;
    d_fparams = d_fparams / f_scale;
    // NaN back-off of TCNNWPFunction::backward (TCNNWP.cpp:231-240), per MLP, dL/dparams and dL/dinput (through what the input
    // gradients feed: d_app / the table gradient).  ExpRunner reads backward_nan_ right after loss.backward(): one host sync.
    Tensor ok_s = torch::isfinite(d_sparams).all();
    if (emb_on) ok_s = ok_s & torch::isfinite(d_app).all();
    Tensor ok_f = torch::isfinite(d_fparams).all() & torch::isfinite(d_table.view({-1}).slice(0, 0, live)).all();
    Tensor flags = torch::stack({ok_s, ok_f}).to(torch::kCPU);
    if (!flags[0].item<bool>()) { shader->global_data_pool_->backward_nan_ = true; shader->mlp_->loss_scale_ = std::max(s_scale / 2.f, 1.f); }
    if (!flags[1].item<bool>()) { field->global_data_pool_->backward_nan_ = true; field->mlp_->loss_scale_ = std::max(f_scale / 2.f, 1.f); }
    return {d_table, d_fparams, d_sparams, emb_on ? d_app : Tensor(), Tensor()};
  }
};

}  // namespace

// =================================================================================================================
RenderResult Renderer::Render(const Tensor& rays_o_raw, const Tensor& rays_d_raw, const Tensor& bounds_raw, const Tensor& emb_idx) {
  if (g_use_reference) return f2b_reference_render(this, rays_o_raw, rays_d_raw, bounds_raw, emb_idx);
  const bool prof_train = global_data_pool_->mode_ == RunningMode::TRAIN;
  ScopedTimer prof_timer(prof_train ? &g_prof.t_render_train : &g_prof.t_render_val, prof_train ? &g_prof.n_train : &g_prof.n_val);
  auto* sampler = dynamic_cast<PersSampler*>(pts_sampler_.get());
  auto* field = dynamic_cast<Hash3DAnchored*>(scene_field_.get());
  auto* shader = dynamic_cast<SHShader*>(shader_.get());
  CHECK(sampler && field && shader) << "B200 Renderer::Render: needs PersSampler + Hash3DAnchored + SHShader";
  CHECK(field->n_hidden_layers_ == 1 && shader->n_hiddens_ == 2) << "B200 Renderer::Render: MLP shapes 32->64->16 / 32->64->64->16 only";
  GlobalDataPool* gdp = global_data_pool_;
  const bool train = gdp->mode_ == RunningMode::TRAIN;
  const int n_rays = rays_o_raw.size(0);
  auto& oct = *sampler->pers_octree_;
  auto main = at::cuda::getCurrentCUDAStream();
  const bool caller_grad = torch::GradMode::is_enabled();                       // ExpRunner's validation paths run under NoGradGuard
  torch::NoGradGuard no_grad;                                                    // everything up to the autograd node is grad-free

  // ---- phase 1: march -> early-stop field pass -> survivor counts, all in the march's slot layout ----------------------
  Tensor rays_o = rays_o_raw.contiguous();
  Tensor rays_d = (rays_d_raw / torch::linalg_norm(rays_d_raw, 2, -1, true)).contiguous();
  Tensor noise;                                                                  // PersSampler.cu:373-381
  if (gdp->mode_ == RunningMode::VALIDATE) noise = torch::ones({kSlot + n_rays + 10}, CUDAFloat);
  else noise = ((torch::rand({kSlot + n_rays + 10}, CUDAFloat) - .5f) + 1.f).contiguous();
  noise.mul_(gdp->ray_march_fineness_);
  Tensor bg;                                                                     // Renderer.cpp:67-81
  if (bg_color_type_ == BGColorType::white) bg = torch::ones({n_rays, 3}, CUDAFloat);
  else if (bg_color_type_ == BGColorType::rand_noise) bg = train ? torch::rand({n_rays, 3}, CUDAFloat) : torch::ones({n_rays, 3}, CUDAFloat) * .5f;
  else bg = torch::zeros({n_rays, 3}, CUDAFloat);
  if (n_rays <= 0) return {bg, torch::zeros({0, 1}, CUDAFloat), torch::zeros({0}, CUDAFloat), Tensor(), torch::zeros({0}, CUDAFloat), Tensor(), Tensor()};

  Work& w = work_of(this);
  w.ensure(n_rays, field->feat_pool_.numel());
  const int local_size = ((field->pool_size_ / N_LEVELS) >> 4) << 4;
  const int64_t live = std::min<int64_t>(field->feat_pool_.numel(), int64_t(N_LEVELS + 1) * local_size);
  // fp16 shadow of the live prefix of the table (the reference re-casts all of it on every AnchoredQuery, Hash3DAnchored.cu:186)
  F2B_CHECK(f2b_table_to_half(field->feat_pool_.data_ptr<float>(), P(w.table16), live, cur_stream()));
  Tensor fparams16 = torch::empty({field->mlp_->params_.numel()}, kHalf);
  F2B_CHECK(f2b_cast_f32_to_f16(field->mlp_->params_.data_ptr<float>(), P(fparams16), fparams16.numel(), 1.f, cur_stream()));
  Tensor counts = torch::empty({n_rays}, CUDAInt), chunk_bounds = torch::empty({n_rays, 2}, CUDAInt);
  Tensor slot_bounds = torch::empty({n_rays, 2}, CUDAInt), first_oct_dis = torch::empty({n_rays, 1}, CUDAFloat);
  Tensor heads = torch::empty({3}, CUDAInt);                                    // [n_kept, n_all, n_all_oct]
  const int n_nodes = oct.tree_nodes_gpu_.numel() / 64, n_trans = oct.pers_trans_gpu_.numel() / 544;
  F2B_CHECK(f2b_sampler_march(P(oct.tree_nodes_gpu_), n_nodes, P(oct.pers_trans_gpu_), n_trans, PF(rays_o), PF(rays_d), PF(noise), n_rays,
                              sampler->global_near_, 1e8f, sampler->sample_l_, sampler->scale_by_dis_ ? 1 : 0,
                              sampler->max_oct_intersect_per_ray_, /*count_all_hits=*/0, PF(w.s_pts), PF(w.s_dt), PF(w.s_t), PI(w.s_anchors),
                              PI(counts), PI(chunk_bounds), PI(heads) + 1, PF(first_oct_dis), cur_stream()));
  F2B_CHECK(f2b_slot_bounds(PI(counts), n_rays, kSlot, 0, PI(slot_bounds), cur_stream()));
  if (!train && fused_forward()) {
    // VALIDATE (ExpRunner::RenderWholeImage / TestImages under NoGradGuard): no gradient, no occupancy votes, no TV-loss edge points.
    // Everything behind the march is ONE kernel walking each ray front to back — encode -> field MLP -> early stop -> SH + shader MLP
    // -> composite — that stops at the first opaque sample (csrc/fused_fwd.cu); values bit-identical to the operator sequence below.
    Tensor sparams16 = torch::empty({shader->mlp_->params_.numel()}, kHalf);
    F2B_CHECK(f2b_cast_f32_to_f16(shader->mlp_->params_.data_ptr<float>(), P(sparams16), sparams16.numel(), 1.f, cur_stream()));
    Tensor colors = torch::empty({n_rays, 3}, CUDAFloat), disp = torch::empty({n_rays}, CUDAFloat), depth = torch::empty({n_rays}, CUDAFloat);
    Tensor kept = torch::empty({n_rays}, CUDAInt), ticket = torch::empty({1}, CUDAInt);
    F2B_CHECK(f2b_render_fwd_fused(P(w.table16), field->prim_pool_.data_ptr<int>(), field->bias_pool_.data_ptr<float>(), field->n_volumes_,
                                   local_size, P(fparams16), P(sparams16), PF(w.s_pts), PF(w.s_dt), PF(w.s_t), PI(w.s_anchors), PI(counts),
                                   PF(rays_d), PF(bg), n_rays, kSlot, PI(heads) + 1, PI(ticket), PF(colors), PF(disp), PF(depth), PI(kept),
                                   PF(w.w0), cur_stream()));
    sample_result_ = SampleResultFlex();
    sample_result_.first_oct_dis = first_oct_dis;
    if (!validate_weights()) return {colors, first_oct_dis, disp, Tensor(), depth, Tensor(), Tensor()};
    // RenderResult.weights / idx_start_end (Renderer.h:24-25) in the reference's packed ray order: one scan, the host read of the
    // survivor total, one gather (nothing on the evaluation path reads them; F2B_VALIDATE_WEIGHTS=0 skips this and the sync)
    Tensor new_bounds = torch::empty({n_rays, 2}, CUDAInt);
    F2B_CHECK(f2b_count_scan(PI(kept), n_rays, PI(new_bounds), PI(heads), cur_stream()));
    Tensor heads_cpu = heads.to(torch::kCPU);
    const int64_t n_kept = heads_cpu[0].item<int>(), n_all = heads_cpu[1].item<int>();
    sample_result_.pts = torch::empty({n_all, 0}, CUDAFloat);
    if (n_all > 0) { burn_mlp_output(n_all); burn_mlp_output(n_kept); burn_mlp_output(n_kept); }   // the three TCNNWP::Query outputs (rng parity)
    Tensor weights = torch::empty({n_kept}, CUDAFloat);
    if (n_kept > 0) F2B_CHECK(f2b_gather_kept_weights(PF(w.w0), PI(new_bounds), n_rays, kSlot, PF(weights), cur_stream()));
    if (n_all <= 0) return {bg, torch::zeros({n_rays, 1}, CUDAFloat), torch::zeros({n_rays}, CUDAFloat), Tensor(), torch::full({n_rays}, 512.f, CUDAFloat), Tensor(), Tensor()};
    return {colors, first_oct_dis, disp, Tensor(), depth, weights, new_bounds};
  }
  F2B_CHECK(f2b_field_fwd_slots(P(w.table16), field->prim_pool_.data_ptr<int>(), field->bias_pool_.data_ptr<float>(), field->n_volumes_,
                                local_size, P(fparams16), PF(w.s_pts), PI(w.s_anchors), 2, PI(counts), n_rays, kSlot, 1, PF(w.logit_s),
                                P(w.feat_s), cur_stream()));
  F2B_CHECK(f2b_early_stop_rays(PF(w.logit_s), 1, PF(w.s_dt), PI(slot_bounds), n_rays, PF(w.w0), PF(w.a0), w.keep.data_ptr<uint8_t>(),
                                PI(w.kept_counts), cur_stream()));
  Tensor new_bounds = torch::empty({n_rays, 2}, CUDAInt);
  F2B_CHECK(f2b_count_scan(PI(w.kept_counts), n_rays, PI(new_bounds), PI(heads), cur_stream()));
  Tensor heads_cpu = heads.to(torch::kCPU);                                      // THE host sync of the step
  const int64_t n_kept = heads_cpu[0].item<int>(), n_all = heads_cpu[1].item<int>(), n_all_oct = heads_cpu[2].item<int>();
  if (gdp->mode_ != RunningMode::VALIDATE)                                       // PersSampler.cu:378-379
    gdp->sampled_oct_per_ray_ = gdp->sampled_oct_per_ray_ * .9f + (float(n_all_oct) / float(n_rays)) * .1f;
  if (train) gdp->sampled_pts_per_ray_ = gdp->sampled_pts_per_ray_ * .9f + (float(n_all) / float(n_rays)) * .1f;
  if (n_all <= 0) {                                                              // Renderer.cpp:83-97
    if (train) gdp->meaningful_sampled_pts_per_ray_ *= .9f;
    return {bg, torch::zeros({n_rays, 1}, CUDAFloat), torch::zeros({n_rays}, CUDAFloat), Tensor(), torch::full({n_rays}, 512.f, CUDAFloat), Tensor(), Tensor()};
  }
  burn_mlp_output(n_all);                                                        // the early-stop AnchoredQuery's torch::rand output

  if (g_keep_samples) {                                                            // Renderer::sample_result_ in the reference's layout (debug / dumps)
    Tensor b = torch::empty({n_rays, 2}, CUDAInt), tot = torch::zeros({1}, CUDAInt);
    F2B_CHECK(f2b_count_scan(PI(counts), n_rays, PI(b), PI(tot), cur_stream()));
    SampleResultFlex s;
    s.pts = torch::empty({n_all, 3}, CUDAFloat); s.dirs = torch::empty({n_all, 3}, CUDAFloat); s.dt = torch::empty({n_all}, CUDAFloat);
    s.t = torch::empty({n_all}, CUDAFloat); s.anchors = torch::empty({n_all, 3}, CUDAInt); s.pts_idx_bounds = b; s.first_oct_dis = first_oct_dis;
    F2B_CHECK(f2b_sampler_gather(PF(rays_d), PI(b), n_rays, PF(w.s_pts), PF(w.s_dt), PF(w.s_t), PI(w.s_anchors), PF(s.pts), PF(s.dirs),
                                 PF(s.dt), PF(s.t), PI(s.anchors), cur_stream()));
    sample_result_ = s;
  } else {                                                                       // not materialised: only the sample COUNT stays readable
    sample_result_ = SampleResultFlex();
    sample_result_.pts = torch::empty({n_all, 0}, CUDAFloat);
    sample_result_.first_oct_dis = first_oct_dis;
  }

  bool votes_on_side = false;
  if (train) {
    // UpdateOctNodes (PersSampler.cu:536-603) on the slot layout.  The votes only feed the NEXT iteration's march: they run on a
    // side stream beside the gradient pass, except on the iterations where the host-side octree maintenance follows at once.
    bool maintenance = gdp->iter_step_ % sampler->compact_freq_ == 0 ||
                       (!sampler->sub_div_milestones_.empty() && sampler->sub_div_milestones_.back() <= gdp->iter_step_);
    Tensor vote_w = torch::full({n_nodes}, -1, CUDAInt), vote_a = torch::full({n_nodes}, -1, CUDAInt), mark = torch::zeros({n_nodes}, CUDAInt);
    auto launch = [&](void* st) {
      F2B_CHECK(f2b_oct_mark_visit(PI(slot_bounds), n_rays, PI(w.s_anchors) + 1, 2, PF(w.w0), PF(w.a0), PI(vote_w), PI(vote_a), PI(mark),
                                   PI(oct.tree_visit_cnt_), st));
      F2B_CHECK(f2b_oct_update_stats(PI(vote_w), PI(vote_a), PI(mark), PI(oct.tree_weight_stats_), PI(oct.tree_alpha_stats_),
                                     P(oct.tree_nodes_gpu_), n_nodes, st));
    };
    if (maintenance) {
      launch(cur_stream());
      while (!sampler->sub_div_milestones_.empty() && sampler->sub_div_milestones_.back() <= gdp->iter_step_) {    // PersSampler.cu:605-614
        oct.ProcOctree(true, true, sampler->sub_div_milestones_.back() <= 0);
        oct.MarkInvisibleNodes();
        oct.ProcOctree(true, false, false);
        sampler->sub_div_milestones_.pop_back();
      }
      if (gdp->iter_step_ % sampler->compact_freq_ == 0) oct.ProcOctree(true, false, false);
    } else {
      stream_wait(*w.side_votes, main);
      {
        c10::cuda::CUDAStreamGuard g(*w.side_votes);
        vote_w.record_stream(*w.side_votes); vote_a.record_stream(*w.side_votes); mark.record_stream(*w.side_votes);
        launch((void*) w.side_votes->stream());
      }
      votes_on_side = true;
    }
    gdp->meaningful_sampled_pts_per_ray_ = gdp->meaningful_sampled_pts_per_ray_ * .9f + (float(n_kept) / float(n_rays)) * .1f;
  }

  // ---- phase 2 inputs: compaction of the survivors (samples + their encoded features), TV-loss edge points ------------
  auto pk = std::make_shared<Pack>();
  Pack& k = *pk;
  k.renderer = this; k.field = field; k.shader = shader;
  const int64_t n_edge = train ? 2 * kEdgePts : 0;
  k.n_kept = n_kept; k.n_edge = n_edge;
  k.feat16 = torch::empty({n_kept + n_edge, 32}, kHalf);
  k.pts = torch::empty({n_kept, 3}, CUDAFloat); k.dirs = torch::empty({n_kept, 3}, CUDAFloat);
  k.dt = torch::empty({n_kept}, CUDAFloat); k.t = torch::empty({n_kept}, CUDAFloat); k.anchors = torch::empty({n_kept, 3}, CUDAInt);
  k.bounds = new_bounds; k.bg = bg;
  F2B_CHECK(f2b_compact_slots(w.keep.data_ptr<uint8_t>(), PI(slot_bounds), PI(new_bounds), n_rays, PF(rays_d), PF(w.s_pts), PF(w.s_dt),
                              PF(w.s_t), PI(w.s_anchors), P(w.feat_s), PF(k.pts), PF(k.dirs), PF(k.dt), PF(k.t), PI(k.anchors), P(k.feat16),
                              cur_stream()));
  if (train) {
    const int n_edges = oct.edge_pool_.size();
    Tensor edge_idx = torch::randint(0, n_edges, {kEdgePts}, CUDAInt).contiguous();                 // PersSampler.cu:456-457
    Tensor edge_coord = (torch::rand({kEdgePts, 2}, CUDAFloat) * 2.f - 1.f).contiguous();
    k.e_pts = torch::empty({kEdgePts * 2, 3}, CUDAFloat); k.e_anc = torch::empty({kEdgePts * 2}, CUDAInt);
    F2B_CHECK(f2b_edge_samples(P(oct.edge_pool_gpu_), P(oct.pers_trans_gpu_), PI(edge_idx), PF(edge_coord), kEdgePts, PF(k.e_pts), PI(k.e_anc),
                               cur_stream()));
    F2B_CHECK(f2b_hash_fwd(P(w.table16), field->prim_pool_.data_ptr<int>(), field->bias_pool_.data_ptr<float>(), field->n_volumes_, local_size,
                           PF(k.e_pts), PI(k.e_anc), 1, (int) n_edge, (char*) P(k.feat16) + n_kept * 64, cur_stream()));
  }
  burn_mlp_output(n_kept + n_edge);                                              // second AnchoredQuery (Renderer.cpp:165/172) ...
  burn_mlp_output(n_kept);                                                       // ... and the shader MLP (SHShader.cpp:27)
  if (train && use_app_emb_) {
    k.ray_emb_idx = emb_idx.to(torch::kInt32).contiguous();
    k.pt_emb_idx = torch::empty({n_kept}, CUDAInt);
    F2B_CHECK(f2b_scatter_idx(PI(new_bounds), PI(k.ray_emb_idx), n_rays, PI(k.pt_emb_idx), cur_stream()));
  }
  k.gs_progress = gdp->gradient_scaling_progress_;
  k.grad_on = caller_grad && train;
  int64_t id;
  {
    std::lock_guard<std::mutex> l(g_pack_mu);
    id = g_pack_next++;
    g_packs[id] = pk;
    for (auto it = g_packs.begin(); it != g_packs.end();)          // a forward whose backward never ran must not pin its activations
      it = (it->first + 4 < id) ? g_packs.erase(it) : std::next(it);
  }
  variable_list out;
  {
    torch::AutoGradMode grad_mode(k.grad_on);
    out = RenderFn::apply(field->feat_pool_, field->mlp_->params_, shader->mlp_->params_, app_emb_, id);
  }
  if (!k.grad_on) { std::lock_guard<std::mutex> l(g_pack_mu); g_packs.erase(id); }
  if (votes_on_side) stream_wait(main, *w.side_votes);                           // joined before w0 / a0 can be recycled
  return {out[0], first_oct_dis, out[1], train ? out[4] : Tensor(), out[2], out[3], new_bounds};
}
