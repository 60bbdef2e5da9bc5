// hash.cuh — device functions of the anchored hash-grid encode and its backward shared by hash.cu (stand-alone encode / scatter),
// field.cu (encode fused in front of the tcgen05 MLP) and mlp_tc_bwd.cu (scatter fused behind the field-MLP backward).
// See hash.cu for the design notes.
#pragma once
#include "common.cuh"

namespace f2b {

__device__ __forceinline__ float level_scale(int l) {
  // exp2f((10-3)*float(l)/15 + 3): cvt(7*l) ; div.rn 15 ; add 3 ; ex2.approx  (Hash3DAnchored.cu:29)
  return exp2f(fadd(fdiv((float)(7 * l), 15.f), 3.f));
}

struct Corner8 {
  unsigned idx[8];   // order 000,001,010,011,100,101,110,111 (z fastest)
  float w[8];
  unsigned cell[3];  // integer cell coordinates (exact run key for the backward's merging)
};

// index/weight computation shared by forward and backward (Hash3DAnchored.cu:27-66)
__device__ __forceinline__ void corners(float x0, float x1, float x2, float scale,
                                        const int* __restrict__ prim, const float* __restrict__ bias,
                                        unsigned local_size, Corner8& c) {
  const float px = ffma(x0, scale, __ldg(bias)), py = ffma(x1, scale, __ldg(bias + 1)),
              pz = ffma(x2, scale, __ldg(bias + 2));
  const float fx = floorf(px), fy = floorf(py), fz = floorf(pz);
  const unsigned ix = (unsigned)fx, iy = (unsigned)fy, iz = (unsigned)fz;   // cvt.rzi.u32.f32 (saturating)
  c.cell[0] = ix; c.cell[1] = iy; c.cell[2] = iz;
  const unsigned pa = (unsigned)__ldg(prim), pb = (unsigned)__ldg(prim + 1), pc = (unsigned)__ldg(prim + 2);
  const unsigned hx0 = ix * pa, hx1 = hx0 + pa, hy0 = iy * pb, hy1 = hy0 + pb, hz0 = iz * pc, hz1 = hz0 + pc;
  const bool pow2 = (local_size & (local_size - 1)) == 0;
  const unsigned mask = local_size - 1;
#define F2B_MOD(v) (pow2 ? ((v) & mask) : ((v) % local_size))
  c.idx[0] = F2B_MOD(hx0 ^ hy0 ^ hz0);
  c.idx[1] = F2B_MOD(hx0 ^ hy0 ^ hz1);
  c.idx[2] = F2B_MOD(hx0 ^ hy1 ^ hz0);
  c.idx[3] = F2B_MOD(hx0 ^ hy1 ^ hz1);
  c.idx[4] = F2B_MOD(hx1 ^ hy0 ^ hz0);
  c.idx[5] = F2B_MOD(hx1 ^ hy0 ^ hz1);
  c.idx[6] = F2B_MOD(hx1 ^ hy1 ^ hz0);
  c.idx[7] = F2B_MOD(hx1 ^ hy1 ^ hz1);
#undef F2B_MOD
  const float a = fsub(px, fx), b = fsub(py, fy), cc = fsub(pz, fz);
  const float na = fsub(1.f, a), nb = fsub(1.f, b), nc = fsub(1.f, cc);
  const float nanb = fmul(na, nb), nab = fmul(na, b), anb = fmul(a, nb), ab = fmul(a, b);
  c.w[0] = fmul(nanb, nc); c.w[1] = fmul(cc, nanb);
  c.w[2] = fmul(nab, nc);  c.w[3] = fmul(nab, cc);
  c.w[4] = fmul(anb, nc);  c.w[5] = fmul(cc, anb);
  c.w[6] = fmul(ab, nc);   c.w[7] = fmul(ab, cc);
}

__device__ __forceinline__ uint32_t ldg_nc_u32(const void* p) {
  uint32_t v;
  asm volatile("ld.global.nc.b32 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}

// Encode one sample at one level: returns the two blended channels packed as half2 bits.
__device__ __forceinline__ uint32_t encode_level(const __half* __restrict__ table, int l, int local_size,
                                                 const Corner8& c) {
  const __half* base = table + size_t(l) * local_size;         // HALF-element offset: levels overlap (quirk)
  uint32_t raw[8];
#pragma unroll
  for (int k = 0; k < 8; k++) raw[k] = ldg_nc_u32(base + size_t(c.idx[k]) * 2);
  float2 f[8];
#pragma unroll
  for (int k = 0; k < 8; k++) f[k] = __half22float2(*reinterpret_cast<const __half2*>(&raw[k]));
  float a0 = fmul(c.w[1], f[1].x), a1 = fmul(c.w[1], f[1].y);
  a0 = ffma(c.w[0], f[0].x, a0); a1 = ffma(c.w[0], f[0].y, a1);
#pragma unroll
  for (int k = 2; k < 8; k++) { a0 = ffma(c.w[k], f[k].x, a0); a1 = ffma(c.w[k], f[k].y, a1); }
  const __half2 h = __floats2half2_rn(a0, a1);
  return *reinterpret_cast<const uint32_t*>(&h);
}

// Encode all 16 levels of one sample into 16 half2 words (registers).  Shared with field.cu.
// `scales` = the 16 level scales computed AT RUN TIME (shared memory): a compile-time-folded exp2f
// would be correctly rounded, MUFU.EX2 (what the reference executes) is not.
__device__ __forceinline__ void encode_point(const __half* __restrict__ table,
                                             const int* __restrict__ prim_pool,
                                             const float* __restrict__ bias_pool, int n_volumes,
                                             int local_size, const float* scales, float p0, float p1,
                                             float p2, int v, uint32_t out[16]) {
  const float x0 = fmul(fadd(p0, 1.f), .5f), x1 = fmul(fadd(p1, 1.f), .5f), x2 = fmul(fadd(p2, 1.f), .5f);
#pragma unroll
  for (int l = 0; l < F2B_N_LEVELS; l++) {
    const int tv = l * n_volumes + v;
    Corner8 c;
    corners(x0, x1, x2, scales[l], prim_pool + tv * 3, bias_pool + tv * 3, (unsigned)local_size, c);
    out[l] = encode_level(table, l, local_size, c);
  }
}

// Backward of one level for a warp that owns 32 CONSECUTIVE samples (lane i = sample i of the group).  Samples of a ray are
// consecutive, so at the coarse levels many lanes fall into the same grid cell and hit the same 8 table entries.  Lanes are grouped
// into runs of identical (cell, volume); when the warp has few runs, the 16 per-run sums (8 corners x 2 channels) are formed with a
// segmented shuffle scan and only the run's last lane issues the 8 vector reductions red.global.add.v2.f32 — up to 32x fewer L2
// atomics at the coarse levels; fine levels (every lane its own run) take the direct path.  fp32 accumulation (the reference
// accumulates fp16 atomics of grad*128, Hash3DAnchored.cu:145-151, and casts/divides afterwards); zero-gradient rows are skipped
// (:149) — a NaN row stays live, so a non-finite gradient still reaches the table.
// (x0, x1, x2) = (pts + 1) / 2 and v = the volume of the lane's sample, read only on live lanes; (g0, g1) = dL/d the level's two
// features, before grad_mul.  Shared by hash_bwd_kernel (hash.cu) and field_bwd_scatter_kernel (mlp_tc_bwd.cu).
constexpr int kDirectHeads = 24;

__device__ __forceinline__ void hash_bwd_level(int l, int lane, bool valid, float x0, float x1, float x2, int v, float g0, float g1,
                                               const int* __restrict__ prim_pool, const float* __restrict__ bias_pool, int n_volumes,
                                               int local_size, float grad_mul, float* __restrict__ grad_table) {
  const bool live = valid && !(g0 == 0.f && g1 == 0.f);
  if (!__any_sync(0xffffffffu, live)) return;
  g0 *= grad_mul; g1 *= grad_mul;
  Corner8 c;
  if (live) {
    const int tv = l * n_volumes + v;
    corners(x0, x1, x2, level_scale(l), prim_pool + tv * 3, bias_pool + tv * 3, (unsigned)local_size, c);
  } else {
#pragma unroll
    for (int k = 0; k < 8; k++) { c.idx[k] = 0; c.w[k] = 0.f; }
    c.cell[0] = c.cell[1] = c.cell[2] = 0;
    v = -1;
  }
  // run heads: key differs from the previous lane (dead lanes never merge)
  const unsigned pcx = __shfl_up_sync(0xffffffffu, c.cell[0], 1), pcy = __shfl_up_sync(0xffffffffu, c.cell[1], 1),
                 pcz = __shfl_up_sync(0xffffffffu, c.cell[2], 1);
  const int prev_v = __shfl_up_sync(0xffffffffu, v, 1);       // dead lanes carry v = -1 and never merge
  const bool head = (lane == 0) || !live || c.cell[0] != pcx || c.cell[1] != pcy || c.cell[2] != pcz || v != prev_v;
  const unsigned heads = __ballot_sync(0xffffffffu, head);
  float* base = grad_table + size_t(l) * local_size;
  if (__popc(heads) > kDirectHeads) {                         // mostly singleton runs: direct reductions
    if (live) {
#pragma unroll
      for (int k = 0; k < 8; k++)
        atomicAdd(reinterpret_cast<float2*>(base + size_t(c.idx[k]) * 2), make_float2(c.w[k] * g0, c.w[k] * g1));
    }
    return;
  }
  // segmented inclusive scan within runs; the last lane of each run holds the run total
  const unsigned below = heads & ((2u << lane) - 1u);         // heads at or below my lane
  const int run_start = 31 - __clz(below);
  float s[16];
#pragma unroll
  for (int k = 0; k < 8; k++) { s[2 * k] = c.w[k] * g0; s[2 * k + 1] = c.w[k] * g1; }
  // only ceil(log2(longest run)) stages move data; the rest would be no-ops (warp-uniform early exit)
  const int max_run = __reduce_max_sync(0xffffffffu, lane - run_start + 1);
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    if (o >= max_run) break;
    const bool take = (lane - o) >= run_start;
#pragma unroll
    for (int k = 0; k < 16; k++) {
      const float u = __shfl_up_sync(0xffffffffu, s[k], o);
      if (take) s[k] += u;
    }
  }
  const bool tail = (lane == 31) || ((heads >> (lane + 1)) & 1u);
  if (live && tail) {
#pragma unroll
    for (int k = 0; k < 8; k++)
      atomicAdd(reinterpret_cast<float2*>(base + size_t(c.idx[k]) * 2), make_float2(s[2 * k], s[2 * k + 1]));
  }
}

}  // namespace f2b
