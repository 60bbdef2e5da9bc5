// hash.cu — anchored multi-level hash-grid encode (forward gather, backward scatter) for sm_100a.
//
// Replaces Hash3DAnchoredForwardKernel / Hash3DAnchoredBackwardKernel
// (src/Field/Hash3DAnchored.cu:11-155) and the per-call dtype passes of
// Hash3DAnchoredFunction::forward/backward (:160-233) and Hash3DAnchored::AnchoredQuery's
// (pts+1)/2 (src/Field/Hash3DAnchored.cpp:91).
//
// B200 design: one thread owns one sample for all 16 levels (the reference launches 16 grid.y
// passes that each re-read the point), lanes of a warp hold 32 consecutive samples of (mostly)
// one ray so the coarse levels' corners coalesce into the same 32 B sectors in L1; the 8 corner
// loads of a level are issued back to back (8-16 independent 4 B half2 gathers in flight per
// thread), the 32 encoded halfs leave as four 128-bit stores.  The fp16 table (17 MB live at
// log2 19) is L2 resident on B200, so the bound is L2->SM sector throughput, not HBM.
// The blend reproduces the reference build's exact fp32 sequence (read off its PTX):
//   acc = w001*f001; acc = fma(w000,f000,acc); then fma in order 010,011,100,101,110,111.
#include "common.cuh"
#include "hash.cuh"
#include <stdlib.h>

namespace f2b {

__global__ void __launch_bounds__(128)
hash_fwd_kernel(const __half* __restrict__ table, const int* __restrict__ prim_pool,
                const float* __restrict__ bias_pool, int n_volumes, int local_size,
                const float* __restrict__ pts, const int* __restrict__ vol, int vol_stride, int n_pts,
                __half* __restrict__ out) {
  __shared__ float s_scale[F2B_N_LEVELS];
  if (threadIdx.x < F2B_N_LEVELS) s_scale[threadIdx.x] = level_scale(threadIdx.x);
  __syncthreads();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_pts) return;
  uint32_t o[16];
  encode_point(table, prim_pool, bias_pool, n_volumes, local_size, s_scale, __ldg(pts + size_t(i) * 3),
               __ldg(pts + size_t(i) * 3 + 1), __ldg(pts + size_t(i) * 3 + 2),
               __ldg(vol + size_t(i) * vol_stride), o);
  uint4* dst = reinterpret_cast<uint4*>(out + size_t(i) * 32);
#pragma unroll
  for (int q = 0; q < 4; q++) dst[q] = make_uint4(o[4 * q], o[4 * q + 1], o[4 * q + 2], o[4 * q + 3]);
}

// Encode of a level range only (out rows keep their [P,32] layout; other levels' columns are not written): used to attribute
// the encode's time to level groups (scripts/level_probe.py, profiles/r02_level_probe.md) and by callers that refresh a subset.
__global__ void __launch_bounds__(128)
hash_fwd_levels_kernel(const __half* __restrict__ table, const int* __restrict__ prim_pool,
                       const float* __restrict__ bias_pool, int n_volumes, int local_size,
                       const float* __restrict__ pts, const int* __restrict__ vol, int vol_stride, int n_pts,
                       int level_lo, int n_levels, __half* __restrict__ out) {
  __shared__ float s_scale[F2B_N_LEVELS];
  if (threadIdx.x < F2B_N_LEVELS) s_scale[threadIdx.x] = level_scale(threadIdx.x);
  __syncthreads();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_pts) return;
  const float p0 = __ldg(pts + size_t(i) * 3), p1 = __ldg(pts + size_t(i) * 3 + 1), p2 = __ldg(pts + size_t(i) * 3 + 2);
  const float x0 = fmul(fadd(p0, 1.f), .5f), x1 = fmul(fadd(p1, 1.f), .5f), x2 = fmul(fadd(p2, 1.f), .5f);
  const int v = __ldg(vol + size_t(i) * vol_stride);
  uint32_t* dst = reinterpret_cast<uint32_t*>(out + size_t(i) * 32);
  for (int l = level_lo; l < level_lo + n_levels; l++) {
    const int tv = l * n_volumes + v;
    Corner8 c;
    corners(x0, x1, x2, s_scale[l], prim_pool + tv * 3, bias_pool + tv * 3, (unsigned)local_size, c);
    dst[l] = encode_level(table, l, local_size, c);
  }
}

// Backward: a warp-task is (32 consecutive samples, one level); the per-level body is hash_bwd_level (hash.cuh).
// The grid is PERSISTENT and bounded (ctas_per_sm x SM count CTAs striding over the (32 samples, level) tasks): a few resident
// warps per SM already saturate the reduction pipe, and a bounded grid lets the scatter of one ray chunk run on a side stream
// next to the tcgen05 kernels of the next chunk without crowding their CTAs out (an unbounded grid of 260 k small blocks did).
template <bool GRAD_F16>
__device__ __forceinline__ void hash_bwd_task(int64_t group, int l, int lane, const int* __restrict__ prim_pool,
                                              const float* __restrict__ bias_pool, int n_volumes, int local_size,
                                              const float* __restrict__ pts, const int* __restrict__ vol, int vol_stride, int n_pts,
                                              const void* __restrict__ grad_feat, float grad_mul, float* __restrict__ grad_table) {
  const int64_t i = group * 32 + lane;
  const bool valid = i < n_pts;
  float g0 = 0.f, g1 = 0.f;
  if (valid) {
    if (GRAD_F16) {
      const float2 gf = __half22float2(reinterpret_cast<const __half2*>(grad_feat)[i * 16 + l]);
      g0 = gf.x; g1 = gf.y;
    } else {
      const float2 gf = reinterpret_cast<const float2*>(grad_feat)[i * 16 + l];
      g0 = gf.x; g1 = gf.y;
    }
  }
  const bool live = valid && !(g0 == 0.f && g1 == 0.f);
  float x0 = 0.f, x1 = 0.f, x2 = 0.f;
  int v = -1;
  if (live) {
    const float p0 = __ldg(pts + i * 3), p1 = __ldg(pts + i * 3 + 1), p2 = __ldg(pts + i * 3 + 2);
    x0 = fmul(fadd(p0, 1.f), .5f); x1 = fmul(fadd(p1, 1.f), .5f); x2 = fmul(fadd(p2, 1.f), .5f);
    v = __ldg(vol + i * vol_stride);
  }
  hash_bwd_level(l, lane, valid, x0, x1, x2, v, g0, g1, prim_pool, bias_pool, n_volumes, local_size, grad_mul, grad_table);
}

template <bool GRAD_F16>
__global__ void __launch_bounds__(256)
hash_bwd_kernel(const int* __restrict__ prim_pool, const float* __restrict__ bias_pool, int n_volumes,
                int local_size, const float* __restrict__ pts, const int* __restrict__ vol,
                int vol_stride, int n_pts, const void* __restrict__ grad_feat, float grad_mul,
                float* __restrict__ grad_table, int64_t n_tasks, int level_lo, int log2_levels) {
  const int lane = threadIdx.x & 31;
  const int64_t stride = (int64_t(gridDim.x) * blockDim.x) >> 5;
  const int lmask = (1 << log2_levels) - 1;
  // A warp would otherwise keep ONE level for all its tasks (the stride is a multiple of the level count) and the fine-level warps
  // (8 reductions per lane, no merging) would finish long after the coarse-level ones: rotate the level by the iteration count —
  // within every stride-sized block of tasks each (32 samples, level) pair is still visited exactly once.
  int k = 0;
  for (int64_t w = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5; w < n_tasks; w += stride, k++)
    hash_bwd_task<GRAD_F16>(w >> log2_levels, level_lo + ((int(w & lmask) + k) & lmask), lane, prim_pool, bias_pool, n_volumes, local_size,
                            pts, vol, vol_stride, n_pts, grad_feat, grad_mul, grad_table);
}

__global__ void level_scales_kernel(float* out) {
  if (threadIdx.x < F2B_N_LEVELS) out[threadIdx.x] = level_scale(threadIdx.x);
}

}  // namespace f2b

using namespace f2b;

extern "C" int f2b_hash_level_scales(float* scales16_host) {
  F2B_REQUIRE(scales16_host, "f2b_hash_level_scales: null pointer");
  float* d = nullptr;
  if (cudaMalloc(&d, 16 * sizeof(float)) != cudaSuccess) { set_error("f2b_hash_level_scales: cudaMalloc failed"); cudaGetLastError(); return F2B_ECUDA; }
  level_scales_kernel<<<1, 32>>>(d);
  cudaError_t e = cudaMemcpy(scales16_host, d, 16 * sizeof(float), cudaMemcpyDeviceToHost);
  cudaFree(d);
  if (e != cudaSuccess) { set_error("f2b_hash_level_scales: %s", cudaGetErrorString(e)); return F2B_ECUDA; }
  return F2B_OK;
}

extern "C" int f2b_hash_fwd(const void* table_f16, const int* prim_pool, const float* bias_pool,
                            int n_volumes, int local_size, const float* pts, const int* vol,
                            int vol_stride, int n_pts, void* out_f16, void* stream) {
  if (n_pts <= 0) return F2B_OK;
  F2B_REQUIRE(table_f16 && prim_pool && bias_pool && pts && vol && out_f16, "f2b_hash_fwd: null pointer");
  F2B_REQUIRE(n_volumes > 0 && local_size > 0 && (local_size % 2) == 0, "f2b_hash_fwd: bad n_volumes/local_size");
  hash_fwd_kernel<<<div_up(n_pts, 128), 128, 0, as_stream(stream)>>>(
      (const __half*)table_f16, prim_pool, bias_pool, n_volumes, local_size, pts, vol, vol_stride, n_pts,
      (__half*)out_f16);
  return check_launch("f2b_hash_fwd");
}

extern "C" int f2b_hash_fwd_levels(const void* table_f16, const int* prim_pool, const float* bias_pool,
                                   int n_volumes, int local_size, const float* pts, const int* vol,
                                   int vol_stride, int n_pts, int level_lo, int n_levels, void* out_f16, void* stream) {
  if (n_pts <= 0) return F2B_OK;
  F2B_REQUIRE(table_f16 && prim_pool && bias_pool && pts && vol && out_f16, "f2b_hash_fwd_levels: null pointer");
  F2B_REQUIRE(n_volumes > 0 && local_size > 0 && (local_size % 2) == 0, "f2b_hash_fwd_levels: bad n_volumes/local_size");
  F2B_REQUIRE(level_lo >= 0 && n_levels > 0 && level_lo + n_levels <= F2B_N_LEVELS, "f2b_hash_fwd_levels: level range outside [0,16)");
  hash_fwd_levels_kernel<<<div_up(n_pts, 128), 128, 0, as_stream(stream)>>>(
      (const __half*)table_f16, prim_pool, bias_pool, n_volumes, local_size, pts, vol, vol_stride, n_pts, level_lo, n_levels,
      (__half*)out_f16);
  return check_launch("f2b_hash_fwd_levels");
}

// Levels [level_lo, level_lo + n_levels) only (n_levels a power of two).  Level l writes the fp32 slab
// [l*local_size, (l+2)*local_size) of grad_table (the half-overlapping level layout, Hash3DAnchored.cu:37), so once the groups
// above and including level l have run, everything from float (l+1)*local_size upwards is final: a data-parallel host launches
// the groups top-down and starts the all-reduce of each finished slab while the next group still scatters (f2nerf_b200/dist.py).
extern "C" int f2b_hash_bwd_levels(const int* prim_pool, const float* bias_pool, int n_volumes, int local_size,
                                   const float* pts, const int* vol, int vol_stride, int n_pts,
                                   const void* grad_feat, int grad_is_f16, float grad_mul, float* grad_table,
                                   int level_lo, int n_levels, void* stream) {
  if (n_pts <= 0) return F2B_OK;
  F2B_REQUIRE(prim_pool && bias_pool && pts && vol && grad_feat && grad_table, "f2b_hash_bwd: null pointer");
  F2B_REQUIRE(n_levels > 0 && (n_levels & (n_levels - 1)) == 0 && level_lo >= 0 && level_lo + n_levels <= F2B_N_LEVELS,
              "f2b_hash_bwd_levels: n_levels must be a power of two and the range inside [0,16)");
  int log2_levels = 0;
  while ((1 << log2_levels) < n_levels) log2_levels++;
  const int64_t n_tasks = int64_t(div_up(n_pts, 32)) * n_levels;           // one warp-task per (32 samples, level)
  static int ctas_per_sm = -1;                                             // resident 256-thread CTAs per SM (F2B_SCATTER_CTAS, default 8 = all)
  if (ctas_per_sm < 0) { const char* e = getenv("F2B_SCATTER_CTAS"); ctas_per_sm = e ? atoi(e) : 8; if (ctas_per_sm < 1) ctas_per_sm = 1; }
  int sms = 148;
  f2b_device_info(&sms, nullptr);
  const int64_t want = div_up(n_tasks * 32, int64_t(256));
  int blocks = int(want < int64_t(sms) * ctas_per_sm ? want : int64_t(sms) * ctas_per_sm);
  // persistent grid: the warp count (8 per block) must be a multiple of n_levels (<= 16) for the kernel's level rotation to visit
  // every task exactly once
  if (blocks < want && ((blocks * 8) % n_levels) != 0) blocks = blocks > 1 ? blocks - 1 : int(want);
  if (grad_is_f16)
    hash_bwd_kernel<true><<<blocks, 256, 0, as_stream(stream)>>>(prim_pool, bias_pool, n_volumes, local_size, pts, vol, vol_stride,
                                                                 n_pts, grad_feat, grad_mul, grad_table, n_tasks, level_lo, log2_levels);
  else
    hash_bwd_kernel<false><<<blocks, 256, 0, as_stream(stream)>>>(prim_pool, bias_pool, n_volumes, local_size, pts, vol, vol_stride,
                                                                  n_pts, grad_feat, grad_mul, grad_table, n_tasks, level_lo, log2_levels);
  return check_launch("f2b_hash_bwd");
}

extern "C" int f2b_hash_bwd(const int* prim_pool, const float* bias_pool, int n_volumes, int local_size,
                            const float* pts, const int* vol, int vol_stride, int n_pts,
                            const void* grad_feat, int grad_is_f16, float grad_mul, float* grad_table,
                            void* stream) {
  return f2b_hash_bwd_levels(prim_pool, bias_pool, n_volumes, local_size, pts, vol, vol_stride, n_pts, grad_feat, grad_is_f16, grad_mul,
                             grad_table, 0, F2B_N_LEVELS, stream);
}
