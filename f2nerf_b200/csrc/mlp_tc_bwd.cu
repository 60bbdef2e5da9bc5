// mlp_tc_bwd.cu — MLP backward on tcgen05 tensor cores (impl 1).
//
// Replaces kernel_mlp_fused_backward (External/tiny-cuda-nn/src/fully_fused_mlp.cu:150-259), the CUTLASS
// dL/dinput GEMM (:832-835) and the three split-K weight-gradient GEMMs on side streams (:785,819,828)
// with ONE persistent kernel per call.  Per 128-sample tile (thread i == sample i == TMEM lane i):
//   activation gradients  dH = dOut.Wout, dH0 = dH1.Wh, dIn = dH0.W0   — UMMA M128, A = K-major tile of the
//       gradient rows, B = the weight matrix used as MN-major operand straight from its row-major layout
//       (no transposed weight copies);
//   weight gradients      dW = dAct^T . Act  — batch-reduction UMMAs with K = the 128 samples of the tile:
//       both operands MN-major views of the very same shared-memory tiles, M = 64 output rows, fp32
//       accumulators that stay resident in TMEM across all tiles of the CTA and are flushed once with
//       atomicAdd at the end (no split-K workspace, no fp16 accumulation, no reduction kernels).
// TMEM columns: [0,64) activation-gradient accumulator, then dW0 (32), dWout^T (16), dWh (64 when NH).
#include "common.cuh"
#include "tc.cuh"
#include "hash.cuh"
#include <stdlib.h>

namespace f2b {
using namespace tc;

constexpr int kBT = 128;   // tile rows

// Shared memory: resident weights, then TWO stages of per-tile operands (double-buffered cp.async prefetch).
// The activation gradients overwrite the activations they mask in place (dH1 over H1, dH0 over H0): every MMA
// that still needs the forward activation as an operand is issued in the step BEFORE the overwrite.
template <int NH>
struct BwdSmem {
  static constexpr int W0 = 0;                              // [64 x 32]  SW64   4 KB   (B operand, MN-major, K = out row)
  static constexpr int WH = 4096;                           // [64 x 64]  SW128  8 KB   (NH only)
  static constexpr int WO = NH ? 12288 : 4096;              // [16 x 64]  SW128  2 KB
  static constexpr int STAGE0 = WO + 2048;
  static constexpr int DO = 0;                              // stage-relative: [128 x 16] SW32   4 KB
  static constexpr int X = 4096;                            //                 [128 x 32] SW64   8 KB
  static constexpr int H0 = 12288;                          //                 [128 x 64] SW128 16 KB (becomes dH0)
  static constexpr int H1 = 28672;                          //                 [128 x 64] SW128 16 KB (becomes dH1; NH only)
  static constexpr int STAGE_BYTES = NH ? 45056 : 28672;
  static constexpr int BAR = STAGE0 + 2 * STAGE_BYTES;
  static constexpr int BYTES = BAR + 64 + 1024;
  static constexpr int TMEM_COLS = NH ? 256 : 128;
  static constexpr int C_ACT = 0, C_GW0 = 64, C_GWO = 96, C_GWH = 128;
};

__device__ __forceinline__ uint32_t pk(float a, float b) {
  const __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&h);
}

// MN-major operand: tile of [k rows][row_bytes] with matching swizzle; k-step = 16 rows
__device__ __forceinline__ uint64_t mnmajor_desc(uint32_t tile, int row_bytes, int k_step) {
  const uint64_t layout = row_bytes == 128 ? kLayoutSW128 : (row_bytes == 64 ? kLayoutSW64 : kLayoutSW32);
  return make_desc(tile + k_step * 16 * row_bytes, 16, 8 * row_bytes, layout);
}

template <int K>
__device__ __forceinline__ void stage_w(const __half* __restrict__ w, int rows, unsigned char* dst) {
  constexpr int chunks = K / 8;
  for (int i = threadIdx.x; i < rows * chunks; i += blockDim.x) {
    const int r = i / chunks, c = i % chunks;
    *reinterpret_cast<uint4*>(dst + (K == 64 ? sw128_off(r, c) : sw64_off(r, c))) = *reinterpret_cast<const uint4*>(w + r * K + c * 8);
  }
}

__device__ __forceinline__ void cp16(uint32_t dst, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}

// One tile's operand rows (dOut 32 B, x 64 B, h0 128 B, h1 128 B per sample; each a contiguous block in global
// memory) -> swizzled tiles of one stage, 16 B per thread and pass, linear sweep = full 128 B lines.
template <int NH>
__device__ __forceinline__ void prefetch_tile(const __half* __restrict__ dout, const __half* __restrict__ in,
                                              const __half* __restrict__ hidden, const __half* __restrict__ hid_last,
                                              int tile, int n_pts, uint32_t stage) {
  using S = BwdSmem<NH>;
  const int rows = min(kBT, n_pts - tile * kBT);
  const size_t t0 = size_t(tile) * kBT;
  const unsigned char* s_do = reinterpret_cast<const unsigned char*>(dout + t0 * 16);
  const unsigned char* s_x = reinterpret_cast<const unsigned char*>(in + t0 * 32);
  const unsigned char* s_h0 = reinterpret_cast<const unsigned char*>(hidden + t0 * 64);
  const unsigned char* s_h1 = reinterpret_cast<const unsigned char*>(hid_last + t0 * 64);
#pragma unroll
  for (int j = 0; j < 2; j++) {
    const int c = threadIdx.x + kBT * j, r = c >> 1;
    const bool ok = r < rows;
    cp16(stage + S::DO + sw32_off(r, c & 1), s_do + (ok ? size_t(c) * 16 : 0), ok ? 16u : 0u);
  }
#pragma unroll
  for (int j = 0; j < 4; j++) {
    const int c = threadIdx.x + kBT * j, r = c >> 2;
    const bool ok = r < rows;
    cp16(stage + S::X + sw64_off(r, c & 3), s_x + (ok ? size_t(c) * 16 : 0), ok ? 16u : 0u);
  }
#pragma unroll
  for (int j = 0; j < 8; j++) {
    const int c = threadIdx.x + kBT * j, r = c >> 3;
    const bool ok = r < rows;
    cp16(stage + S::H0 + sw128_off(r, c & 7), s_h0 + (ok ? size_t(c) * 16 : 0), ok ? 16u : 0u);
    if (NH) cp16(stage + S::H1 + sw128_off(r, c & 7), s_h1 + (ok ? size_t(c) * 16 : 0), ok ? 16u : 0u);
  }
}

// masked epilogue: acc (64 fp32 from TMEM) * [h > 0] -> fp16 row of the dH tile (SW128)
__device__ __forceinline__ void relu_bwd_epilogue(uint32_t tmem_row, const unsigned char* h_tile, unsigned char* dh_tile, int row) {
#pragma unroll
  for (int q = 0; q < 4; q++) {
    uint32_t r[16];
    tmem_ld16(tmem_row + 16 * q, r);
    tmem_ld_wait();
    uint4 hv[2], o[2];
    hv[0] = *reinterpret_cast<const uint4*>(h_tile + sw128_off(row, 2 * q));
    hv[1] = *reinterpret_cast<const uint4*>(h_tile + sw128_off(row, 2 * q + 1));
    const __half2* hh = reinterpret_cast<const __half2*>(hv);
    uint32_t* ow = reinterpret_cast<uint32_t*>(o);
#pragma unroll
    for (int e = 0; e < 8; e++) {
      const float2 hf = __half22float2(hh[e]);
      ow[e] = pk(hf.x > 0.f ? __uint_as_float(r[2 * e]) : 0.f, hf.y > 0.f ? __uint_as_float(r[2 * e + 1]) : 0.f);
    }
    *reinterpret_cast<uint4*>(dh_tile + sw128_off(row, 2 * q)) = o[0];
    *reinterpret_cast<uint4*>(dh_tile + sw128_off(row, 2 * q + 1)) = o[1];
  }
}

template <int NH>
__global__ void __launch_bounds__(kBT)
mlp_bwd_tc_kernel(const __half* __restrict__ dout, const __half* __restrict__ in, const __half* __restrict__ hidden,
                  const __half* __restrict__ hid_last, const __half* __restrict__ params, int n_pts,
                  __half* __restrict__ din, float* __restrict__ dparams) {
  using S = BwdSmem<NH>;
  extern __shared__ unsigned char smem_raw[];
  unsigned char* sm = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* mbar = reinterpret_cast<uint64_t*>(sm + S::BAR);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sm + S::BAR + 8);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n_tiles = (n_pts + kBT - 1) / kBT;
  const uint32_t stage0 = smem_u32(sm + S::STAGE0);

  int tile = blockIdx.x;
  if (tile < n_tiles) prefetch_tile<NH>(dout, in, hidden, hid_last, tile, n_pts, stage0);
  asm volatile("cp.async.commit_group;" ::: "memory");
  stage_w<32>(params, 64, sm + S::W0);
  if (NH) stage_w<64>(params + 64 * 32, 64, sm + S::WH);
  stage_w<64>(params + 64 * 32 + NH * 64 * 64, 16, sm + S::WO);
  if (tid == 0) mbar_init(mbar, 1);
  if (warp == 0) tmem_alloc(tmem_slot, S::TMEM_COLS);
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = *tmem_slot;
  const uint32_t tmem_row = tmem + (uint32_t(warp * 32) << 16);
  const uint32_t s_w0 = smem_u32(sm + S::W0), s_wh = smem_u32(sm + S::WH), s_wo = smem_u32(sm + S::WO);
  // instruction descriptors
  constexpr uint32_t id_act64 = idesc_f16_f32(128, 64, 0, 1);     // A K-major, B MN-major
  constexpr uint32_t id_act32 = idesc_f16_f32(128, 32, 0, 1);
  constexpr uint32_t id_gw16 = idesc_f16_f32(64, 16, 1, 1);       // both MN-major
  constexpr uint32_t id_gw32 = idesc_f16_f32(64, 32, 1, 1);
  constexpr uint32_t id_gw64 = idesc_f16_f32(64, 64, 1, 1);
  uint32_t phase = 0, first = 1, buf = 0;

  for (; tile < n_tiles; tile += gridDim.x, buf ^= 1) {
    const int p = tile * kBT + tid;
    const bool valid = p < n_pts;
    const int next = tile + gridDim.x;
    if (next < n_tiles) prefetch_tile<NH>(dout, in, hidden, hid_last, next, n_pts, stage0 + (buf ^ 1) * S::STAGE_BYTES);
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 1;" ::: "memory");         // this tile's operands have landed
    fence_async_smem();
    fence_before_sync();
    __syncthreads();
    unsigned char* const st = sm + S::STAGE0 + buf * S::STAGE_BYTES;
    const uint32_t sb = stage0 + buf * S::STAGE_BYTES;
    const uint32_t s_do = sb + S::DO, s_x = sb + S::X, s_h0 = sb + S::H0, s_h1 = sb + S::H1;
    const uint32_t s_hl = NH ? s_h1 : s_h0;
    const uint32_t acc = (first ^ 1);
    // ---- A: dH_last = dOut . Wout  (K = 16) ; dWout^T += H_last^T . dOut (needs H_last before it is overwritten)
    if (tid == 0) {
      fence_after_sync();
      mma_f16(tmem + S::C_ACT, kmajor_desc(s_do, 32), mnmajor_desc(s_wo, 128, 0), id_act64, 0);
#pragma unroll
      for (int k = 0; k < 8; k++)
        mma_f16(tmem + S::C_GWO, mnmajor_desc(s_hl, 128, k), mnmajor_desc(s_do, 32, k), id_gw16, (k > 0) | acc);
      mma_commit(mbar);
    }
    mbar_wait(mbar, phase); phase ^= 1;
    fence_after_sync();
    relu_bwd_epilogue(tmem_row + S::C_ACT, st + (NH ? S::H1 : S::H0), st + (NH ? S::H1 : S::H0), tid);   // in place
    fence_before_sync();
    fence_async_smem();
    __syncthreads();
    if (NH) {
      // ---- B: dH0 = dH1 . Wh ; dWh += dH1^T . H0 (H0 still the forward activation) ---------------------
      if (tid == 0) {
        fence_after_sync();
#pragma unroll
        for (int k = 0; k < 4; k++)
          mma_f16(tmem + S::C_ACT, kmajor_desc(s_h1 + 32 * k, 128), mnmajor_desc(s_wh, 128, k), id_act64, k);
#pragma unroll
        for (int k = 0; k < 8; k++)
          mma_f16(tmem + S::C_GWH, mnmajor_desc(s_h1, 128, k), mnmajor_desc(s_h0, 128, k), id_gw64, (k > 0) | acc);
        mma_commit(mbar);
      }
      mbar_wait(mbar, phase); phase ^= 1;
      fence_after_sync();
      relu_bwd_epilogue(tmem_row + S::C_ACT, st + S::H0, st + S::H0, tid);                                  // in place
      fence_before_sync();
      fence_async_smem();
      __syncthreads();
    }
    // ---- C: dIn = dH0 . W0 ; dW0 += dH0^T . X -----------------------------------------------------------
    if (tid == 0) {
      fence_after_sync();
#pragma unroll
      for (int k = 0; k < 4; k++)
        mma_f16(tmem + S::C_ACT, kmajor_desc(s_h0 + 32 * k, 128), mnmajor_desc(s_w0, 64, k), id_act32, k);
#pragma unroll
      for (int k = 0; k < 8; k++)
        mma_f16(tmem + S::C_GW0, mnmajor_desc(s_h0, 128, k), mnmajor_desc(s_x, 64, k), id_gw32, (k > 0) | acc);
      mma_commit(mbar);
    }
    first = 0;
    mbar_wait(mbar, phase); phase ^= 1;
    fence_after_sync();
    {
#pragma unroll
      for (int q = 0; q < 2; q++) {
        uint32_t r[16];
        tmem_ld16(tmem_row + S::C_ACT + 16 * q, r);
        tmem_ld_wait();
        if (din && valid) {
          uint4 o[2];
          uint32_t* ow = reinterpret_cast<uint32_t*>(o);
#pragma unroll
          for (int e = 0; e < 8; e++) ow[e] = pk(__uint_as_float(r[2 * e]), __uint_as_float(r[2 * e + 1]));
          uint4* dst = reinterpret_cast<uint4*>(din + size_t(p) * 32) + 2 * q;
          dst[0] = o[0]; dst[1] = o[1];
        }
      }
    }
    // the next iteration's barrier orders these TMEM reads before the next tile's first MMA
  }
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  fence_before_sync();
  __syncthreads();
  // ---- flush the weight-gradient accumulators (M = 64 layout: warp w, lanes 0..15 hold rows 16w..16w+15) ----
  if (!first) {
    fence_after_sync();
    const int row = warp * 16 + lane;
    float* g0 = dparams;
    float* gh = dparams + 64 * 32;
    float* go = gh + NH * 64 * 64;
#pragma unroll
    for (int q = 0; q < 2; q++) {
      uint32_t r[16];
      tmem_ld16(tmem_row + S::C_GW0 + 16 * q, r);
      tmem_ld_wait();
      if (lane < 16)
#pragma unroll
        for (int e = 0; e < 16; e++) atomicAdd(g0 + row * 32 + 16 * q + e, __uint_as_float(r[e]));
    }
    {
      uint32_t r[16];
      tmem_ld16(tmem_row + S::C_GWO, r);
      tmem_ld_wait();
      if (lane < 16)
#pragma unroll
        for (int e = 0; e < 16; e++) atomicAdd(go + e * 64 + row, __uint_as_float(r[e]));      // transposed back
    }
    if (NH) {
#pragma unroll
      for (int q = 0; q < 4; q++) {
        uint32_t r[16];
        tmem_ld16(tmem_row + S::C_GWH + 16 * q, r);
        tmem_ld_wait();
        if (lane < 16)
#pragma unroll
          for (int e = 0; e < 16; e++) atomicAdd(gh + row * 64 + 16 * q + e, __uint_as_float(r[e]));
      }
    }
    fence_before_sync();
  }
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, S::TMEM_COLS);
}


// ---------------------------------------------------------------------------------------------------------------------
// Recompute variant (hidden0 == NULL in f2b_mlp_bwd2): the forward pass saves NO hidden activations — 128 B (field) /
// 256 B (shader) per sample it no longer writes and this kernel no longer reads.  The tile's activations are rebuilt on
// the tensor pipe from the 64 B input row (same UMMAs, same operands, same fp16 rounding as mlp_fwd_tc_kernel => the
// very same bits the forward would have saved), then the backward proceeds as above.  r01 profile: these kernels were
// HBM-bound at 0.6-0.87 of peak with the tensor pipe 6-19 % busy — the recompute rides on idle MMA issue slots.
// Per sample: 32 (dOut) + 64 (x) B read, 64 B written  (was 224 / 352 B read).
//   NH = 0:  F0  H0 = relu(X.W0^T)                                  -> H0 tile
//            A   dH0 = (dOut.Wout) * [H0 > 0] ; dWout^T += H0^T.dOut -> dH0 over H0
//            C   dX = dH0.W0 ; dW0 += dH0^T.X
//   NH = 1:  F0  H0 = relu(X.W0^T)  and, into a second accumulator,  G = dOut.Wout   (independent of F0: one round trip)
//            F1  H1 = relu(H0.Wh^T) -> H1 tile ;  dH1 = G * [H1 > 0]  -> D1 tile   (same epilogue, both rows in registers)
//            B   dWout^T += H1^T.dOut ; dH0 = (dH1.Wh) * [H0 > 0] ; dWh += dH1^T.H0 -> dH0 over H0
//            C   dX = dH0.W0 ; dW0 += dH0^T.X
template <int NH>
struct RcSmem {
  static constexpr int W0 = 0;                              // [64 x 32]  SW64   4 KB  (K-major for the forward, MN-major view for the backward)
  static constexpr int WH = 4096;                           // [64 x 64]  SW128  8 KB  (NH only)
  static constexpr int WO = NH ? 12288 : 4096;              // [16 x 64]  SW128  2 KB
  static constexpr int H0 = WO + 2048;                      // [128 x 64] SW128 16 KB  forward H0, then dH0
  static constexpr int H1 = H0 + 16384;                     // [128 x 64] SW128 16 KB  forward H1            (NH only)
  static constexpr int D1 = H1 + 16384;                     // [128 x 64] SW128 16 KB  dH1                   (NH only)
  static constexpr int STAGE0 = NH ? D1 + 16384 : H0 + 16384;
  static constexpr int DO = 0;                              // stage-relative: [128 x 16] SW32 4 KB
  static constexpr int X = 4096;                            //                 [128 x 32] SW64 8 KB
  static constexpr int STAGE_BYTES = 12288;
  static constexpr int BAR = STAGE0 + 2 * STAGE_BYTES;
  static constexpr int BYTES = BAR + 64 + 1024;
  static constexpr int TMEM_COLS = NH ? 256 : 128;
  static constexpr int C_ACT = 0, C_GW0 = 64, C_GWO = 96, C_GWH = 128, C_ACT2 = 192;
};

// operand rows of one tile: dOut [rows,16] and x [rows,32] from the tile's first row on (rows <= kBT; the rest read as zeros)
template <int NH>
__device__ __forceinline__ void prefetch_tile_rc(const __half* __restrict__ dout, const __half* __restrict__ in, int rows, uint32_t stage) {
  using S = RcSmem<NH>;
  const unsigned char* s_do = reinterpret_cast<const unsigned char*>(dout);
  const unsigned char* s_x = reinterpret_cast<const unsigned char*>(in);
#pragma unroll
  for (int j = 0; j < 2; j++) {
    const int c = threadIdx.x + kBT * j, r = c >> 1;
    const bool ok = r < rows;
    cp16(stage + S::DO + sw32_off(r, c & 1), s_do + (ok ? size_t(c) * 16 : 0), ok ? 16u : 0u);
  }
#pragma unroll
  for (int j = 0; j < 4; j++) {
    const int c = threadIdx.x + kBT * j, r = c >> 2;
    const bool ok = r < rows;
    cp16(stage + S::X + sw64_off(r, c & 3), s_x + (ok ? size_t(c) * 16 : 0), ok ? 16u : 0u);
  }
}

// forward epilogue: acc (64 fp32) -> ReLU -> fp16 -> my row of the H tile
__device__ __forceinline__ void relu_fwd_epilogue(uint32_t tmem_row, unsigned char* h_tile, int row) {
#pragma unroll
  for (int q = 0; q < 4; q++) {
    uint32_t r[16];
    tmem_ld16(tmem_row + 16 * q, r);
    tmem_ld_wait();
    uint4 o[2];
    uint32_t* ow = reinterpret_cast<uint32_t*>(o);
#pragma unroll
    for (int e = 0; e < 8; e++) ow[e] = pk(fmaxf(__uint_as_float(r[2 * e]), 0.f), fmaxf(__uint_as_float(r[2 * e + 1]), 0.f));
    *reinterpret_cast<uint4*>(h_tile + sw128_off(row, 2 * q)) = o[0];
    *reinterpret_cast<uint4*>(h_tile + sw128_off(row, 2 * q + 1)) = o[1];
  }
}

// forward + masked-gradient epilogue: h = fp16(relu(acc)) -> H tile ; g * [h > 0] -> fp16 -> D tile (the mask tests the ROUNDED
// activation, like relu_bwd_epilogue reading the saved fp16 tile)
__device__ __forceinline__ void relu_fwd_mask_epilogue(uint32_t tmem_h, uint32_t tmem_g, unsigned char* h_tile, unsigned char* d_tile, int row) {
#pragma unroll
  for (int q = 0; q < 4; q++) {
    uint32_t r[16], g[16];
    tmem_ld16(tmem_h + 16 * q, r);
    tmem_ld16(tmem_g + 16 * q, g);
    tmem_ld_wait();
    uint4 o[2], d[2];
    uint32_t* ow = reinterpret_cast<uint32_t*>(o);
    uint32_t* dw = reinterpret_cast<uint32_t*>(d);
#pragma unroll
    for (int e = 0; e < 8; e++) {
      const __half2 h = __floats2half2_rn(fmaxf(__uint_as_float(r[2 * e]), 0.f), fmaxf(__uint_as_float(r[2 * e + 1]), 0.f));
      ow[e] = *reinterpret_cast<const uint32_t*>(&h);
      const float2 hf = __half22float2(h);
      dw[e] = pk(hf.x > 0.f ? __uint_as_float(g[2 * e]) : 0.f, hf.y > 0.f ? __uint_as_float(g[2 * e + 1]) : 0.f);
    }
    *reinterpret_cast<uint4*>(h_tile + sw128_off(row, 2 * q)) = o[0];
    *reinterpret_cast<uint4*>(h_tile + sw128_off(row, 2 * q + 1)) = o[1];
    *reinterpret_cast<uint4*>(d_tile + sw128_off(row, 2 * q)) = d[0];
    *reinterpret_cast<uint4*>(d_tile + sw128_off(row, 2 * q + 1)) = d[1];
  }
}

template <int NH>
__global__ void __launch_bounds__(kBT)
mlp_bwd_rc_kernel(const __half* __restrict__ dout, const __half* __restrict__ in, const __half* __restrict__ params, int n_pts,
                  __half* __restrict__ din, float* __restrict__ dparams) {
  using S = RcSmem<NH>;
  extern __shared__ unsigned char smem_raw[];
  unsigned char* sm = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* mbar = reinterpret_cast<uint64_t*>(sm + S::BAR);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sm + S::BAR + 8);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n_tiles = (n_pts + kBT - 1) / kBT;
  const uint32_t stage0 = smem_u32(sm + S::STAGE0);

  int tile = blockIdx.x;
  if (tile < n_tiles) prefetch_tile_rc<NH>(dout + size_t(tile) * kBT * 16, in + size_t(tile) * kBT * 32, min(kBT, n_pts - tile * kBT), stage0);
  asm volatile("cp.async.commit_group;" ::: "memory");
  stage_w<32>(params, 64, sm + S::W0);
  if (NH) stage_w<64>(params + 64 * 32, 64, sm + S::WH);
  stage_w<64>(params + 64 * 32 + NH * 64 * 64, 16, sm + S::WO);
  if (tid == 0) mbar_init(mbar, 1);
  if (warp == 0) tmem_alloc(tmem_slot, S::TMEM_COLS);
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = *tmem_slot;
  const uint32_t tmem_row = tmem + (uint32_t(warp * 32) << 16);
  const uint32_t s_w0 = smem_u32(sm + S::W0), s_wh = smem_u32(sm + S::WH), s_wo = smem_u32(sm + S::WO);
  const uint32_t s_h0 = smem_u32(sm + S::H0), s_h1 = smem_u32(sm + S::H1), s_d1 = smem_u32(sm + S::D1);
  constexpr uint32_t id_fwd64 = idesc_f16_f32(128, 64);           // forward layers: both operands K-major
  constexpr uint32_t id_act64 = idesc_f16_f32(128, 64, 0, 1);     // A K-major, B MN-major
  constexpr uint32_t id_act32 = idesc_f16_f32(128, 32, 0, 1);
  constexpr uint32_t id_gw16 = idesc_f16_f32(64, 16, 1, 1);       // both MN-major
  constexpr uint32_t id_gw32 = idesc_f16_f32(64, 32, 1, 1);
  constexpr uint32_t id_gw64 = idesc_f16_f32(64, 64, 1, 1);
  uint32_t phase = 0, first = 1, buf = 0;

  for (; tile < n_tiles; tile += gridDim.x, buf ^= 1) {
    const int p = tile * kBT + tid;
    const bool valid = p < n_pts;
    const int next = tile + gridDim.x;
    if (next < n_tiles)
      prefetch_tile_rc<NH>(dout + size_t(next) * kBT * 16, in + size_t(next) * kBT * 32, min(kBT, n_pts - next * kBT),
                           stage0 + (buf ^ 1) * S::STAGE_BYTES);
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 1;" ::: "memory");         // this tile's operands have landed
    fence_async_smem();
    fence_before_sync();
    __syncthreads();
    const uint32_t sb = stage0 + buf * S::STAGE_BYTES;
    const uint32_t s_do = sb + S::DO, s_x = sb + S::X;
    const uint32_t acc = (first ^ 1);
    // ---- F0: H0 = relu(X . W0^T)   (NH: and G = dOut . Wout into the second accumulator) ----------------
    if (tid == 0) {
      fence_after_sync();
#pragma unroll
      for (int k = 0; k < 2; k++) mma_f16(tmem + S::C_ACT, kmajor_desc(s_x + 32 * k, 64), kmajor_desc(s_w0 + 32 * k, 64), id_fwd64, k);
      if (NH) mma_f16(tmem + S::C_ACT2, kmajor_desc(s_do, 32), mnmajor_desc(s_wo, 128, 0), id_act64, 0);
      mma_commit(mbar);
    }
    mbar_wait(mbar, phase); phase ^= 1;
    fence_after_sync();
    relu_fwd_epilogue(tmem_row + S::C_ACT, sm + S::H0, tid);
    fence_before_sync();
    fence_async_smem();
    __syncthreads();
    if (NH) {
      // ---- F1: H1 = relu(H0 . Wh^T) ; dH1 = G * [H1 > 0] ------------------------------------------------
      if (tid == 0) {
        fence_after_sync();
#pragma unroll
        for (int k = 0; k < 4; k++) mma_f16(tmem + S::C_ACT, kmajor_desc(s_h0 + 32 * k, 128), kmajor_desc(s_wh + 32 * k, 128), id_fwd64, k);
        mma_commit(mbar);
      }
      mbar_wait(mbar, phase); phase ^= 1;
      fence_after_sync();
      relu_fwd_mask_epilogue(tmem_row + S::C_ACT, tmem_row + S::C_ACT2, sm + S::H1, sm + S::D1, tid);
      fence_before_sync();
      fence_async_smem();
      __syncthreads();
      // ---- B: dWout^T += H1^T . dOut ; dH0 = dH1 . Wh ; dWh += dH1^T . H0 (H0 still the forward activation) ----
      if (tid == 0) {
        fence_after_sync();
#pragma unroll
        for (int k = 0; k < 8; k++)
          mma_f16(tmem + S::C_GWO, mnmajor_desc(s_h1, 128, k), mnmajor_desc(s_do, 32, k), id_gw16, (k > 0) | acc);
#pragma unroll
        for (int k = 0; k < 4; k++)
          mma_f16(tmem + S::C_ACT, kmajor_desc(s_d1 + 32 * k, 128), mnmajor_desc(s_wh, 128, k), id_act64, k);
#pragma unroll
        for (int k = 0; k < 8; k++)
          mma_f16(tmem + S::C_GWH, mnmajor_desc(s_d1, 128, k), mnmajor_desc(s_h0, 128, k), id_gw64, (k > 0) | acc);
        mma_commit(mbar);
      }
    } else {
      // ---- A: dH0 = dOut . Wout ; dWout^T += H0^T . dOut -------------------------------------------------
      if (tid == 0) {
        fence_after_sync();
        mma_f16(tmem + S::C_ACT, kmajor_desc(s_do, 32), mnmajor_desc(s_wo, 128, 0), id_act64, 0);
#pragma unroll
        for (int k = 0; k < 8; k++)
          mma_f16(tmem + S::C_GWO, mnmajor_desc(s_h0, 128, k), mnmajor_desc(s_do, 32, k), id_gw16, (k > 0) | acc);
        mma_commit(mbar);
      }
    }
    mbar_wait(mbar, phase); phase ^= 1;
    fence_after_sync();
    relu_bwd_epilogue(tmem_row + S::C_ACT, sm + S::H0, sm + S::H0, tid);                                    // dH0 over H0, in place
    fence_before_sync();
    fence_async_smem();
    __syncthreads();
    // ---- C: dIn = dH0 . W0 ; dW0 += dH0^T . X -----------------------------------------------------------
    if (tid == 0) {
      fence_after_sync();
#pragma unroll
      for (int k = 0; k < 4; k++)
        mma_f16(tmem + S::C_ACT, kmajor_desc(s_h0 + 32 * k, 128), mnmajor_desc(s_w0, 64, k), id_act32, k);
#pragma unroll
      for (int k = 0; k < 8; k++)
        mma_f16(tmem + S::C_GW0, mnmajor_desc(s_h0, 128, k), mnmajor_desc(s_x, 64, k), id_gw32, (k > 0) | acc);
      mma_commit(mbar);
    }
    first = 0;
    mbar_wait(mbar, phase); phase ^= 1;
    fence_after_sync();
#pragma unroll
    for (int q = 0; q < 2; q++) {
      uint32_t r[16];
      tmem_ld16(tmem_row + S::C_ACT + 16 * q, r);
      tmem_ld_wait();
      if (din && valid) {
        uint4 o[2];
        uint32_t* ow = reinterpret_cast<uint32_t*>(o);
#pragma unroll
        for (int e = 0; e < 8; e++) ow[e] = pk(__uint_as_float(r[2 * e]), __uint_as_float(r[2 * e + 1]));
        uint4* dst = reinterpret_cast<uint4*>(din + size_t(p) * 32) + 2 * q;
        dst[0] = o[0]; dst[1] = o[1];
      }
    }
    // the next iteration's barrier orders these TMEM reads before the next tile's first MMA
  }
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  fence_before_sync();
  __syncthreads();
  // ---- flush the weight-gradient accumulators (M = 64 layout: warp w, lanes 0..15 hold rows 16w..16w+15) ----
  if (!first) {
    fence_after_sync();
    const int row = warp * 16 + lane;
    float* g0 = dparams;
    float* gh = dparams + 64 * 32;
    float* go = gh + NH * 64 * 64;
#pragma unroll
    for (int q = 0; q < 2; q++) {
      uint32_t r[16];
      tmem_ld16(tmem_row + S::C_GW0 + 16 * q, r);
      tmem_ld_wait();
      if (lane < 16)
#pragma unroll
        for (int e = 0; e < 16; e++) atomicAdd(g0 + row * 32 + 16 * q + e, __uint_as_float(r[e]));
    }
    {
      uint32_t r[16];
      tmem_ld16(tmem_row + S::C_GWO, r);
      tmem_ld_wait();
      if (lane < 16)
#pragma unroll
        for (int e = 0; e < 16; e++) atomicAdd(go + e * 64 + row, __uint_as_float(r[e]));      // transposed back
    }
    if (NH) {
#pragma unroll
      for (int q = 0; q < 4; q++) {
        uint32_t r[16];
        tmem_ld16(tmem_row + S::C_GWH + 16 * q, r);
        tmem_ld_wait();
        if (lane < 16)
#pragma unroll
          for (int e = 0; e < 16; e++) atomicAdd(gh + row * 64 + 16 * q + e, __uint_as_float(r[e]));
      }
    }
    fence_before_sync();
  }
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, S::TMEM_COLS);
}


// ---------------------------------------------------------------------------------------------------------------------
// Field-MLP backward + hash-table scatter in ONE persistent kernel (f2b_field_bwd_scatter).  The two-kernel sequence
// (mlp_bwd_rc_kernel<0> -> dfeat16 in HBM -> hash_bwd_kernel) rounds dL/dfeatures to fp16, writes it (64 B per row) and reads
// it back, and the scatter reloads the point and its volume once per (sample, level) pair.  Here the dL/dfeatures of a tile go
// from TMEM through shared memory straight to the scatter warps of the same CTA:
//   warps 0-3 (tensor warps, TMEM lanes 0-127)  F0, A, C of mlp_bwd_rc_kernel<0> — same UMMAs, same operands, dW0 / dWout^T
//       resident in TMEM and flushed once; C's epilogue rounds dX with the same pk() into a 2-slot ring (full / empty mbarriers)
//   SCATTER_WARPS further warps                  warp w takes rows [32 (w % 4), 32 (w % 4) + 32) of every (SCATTER_WARPS / 4)-th
//       tile of the CTA, reads each row's point and volume once and walks the 16 levels through hash_bwd_level (hash.cuh).
// Tiles never straddle the ray-sample / edge-point boundary (the edge segment starts a new tile), so a scatter warp's 32 rows are
// exactly a group hash_bwd_kernel forms: the per-run sums are bit-identical, only the order of the fp32 reductions differs.
// Ring: one slot per group of 4 scatter warps (at least two), each [16 levels][128 rows] half2 words (conflict-free both ways).
template <int SCATTER_WARPS>
struct FbsSmem {
  using R = RcSmem<0>;
  static constexpr int SLOTS = SCATTER_WARPS / 4 < 2 ? 2 : SCATTER_WARPS / 4;
  static constexpr int RING = R::BAR;
  static constexpr int SLOT_WORDS = F2B_N_LEVELS * kBT;
  static constexpr int BAR = RING + SLOTS * SLOT_WORDS * 4;  // mma, full[SLOTS], empty[SLOTS], TMEM address
  static constexpr int BYTES = BAR + 16 * (SLOTS + 1) + 1024;
  static constexpr int TMEM_COLS = R::TMEM_COLS;
};

__device__ __forceinline__ void tensor_bar() { asm volatile("bar.sync 1, 128;" ::: "memory"); }   // warps 0-3 only

// dW0 / dWout^T accumulators (M = 64 layout: warp w, lanes 0..15 hold rows 16w..16w+15) -> dparams (atomics)
__device__ __forceinline__ void flush_field_wgrad(uint32_t tmem_row, int warp, int lane, float* __restrict__ dparams) {
  using S = RcSmem<0>;
  const int row = warp * 16 + lane;
  float* g0 = dparams;
  float* go = dparams + 64 * 32;
#pragma unroll
  for (int q = 0; q < 2; q++) {
    uint32_t r[16];
    tmem_ld16(tmem_row + S::C_GW0 + 16 * q, r);
    tmem_ld_wait();
    if (lane < 16)
#pragma unroll
      for (int e = 0; e < 16; e++) atomicAdd(g0 + row * 32 + 16 * q + e, __uint_as_float(r[e]));
  }
  uint32_t r[16];
  tmem_ld16(tmem_row + S::C_GWO, r);
  tmem_ld_wait();
  if (lane < 16)
#pragma unroll
    for (int e = 0; e < 16; e++) atomicAdd(go + e * 64 + row, __uint_as_float(r[e]));      // transposed back
}

template <int SCATTER_WARPS, int MIN_CTAS>
__global__ void __launch_bounds__(kBT + 32 * SCATTER_WARPS, MIN_CTAS)
field_bwd_scatter_kernel(const __half* __restrict__ dout, const __half* __restrict__ in, const __half* __restrict__ params,
                         int n_kept, const float* __restrict__ pts, const int* __restrict__ anchors, int n_edge,
                         const float* __restrict__ e_pts, const int* __restrict__ e_anc, const int* __restrict__ prim_pool,
                         const float* __restrict__ bias_pool, int n_volumes, int local_size, float grad_mul,
                         float* __restrict__ dparams, float* __restrict__ grad_table, int flush_every) {
  static_assert(SCATTER_WARPS % 4 == 0, "a tile's 128 rows are four 32-row scatter groups");
  using S = RcSmem<0>;
  using F = FbsSmem<SCATTER_WARPS>;
  extern __shared__ unsigned char smem_raw[];
  unsigned char* sm = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* mbar = reinterpret_cast<uint64_t*>(sm + F::BAR);
  uint64_t* full = mbar + 1;
  uint64_t* empty = full + F::SLOTS;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(empty + F::SLOTS);
  uint32_t* ring = reinterpret_cast<uint32_t*>(sm + F::RING);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int tiles_k = (n_kept + kBT - 1) / kBT;
  const int n_tiles = tiles_k + (n_edge + kBT - 1) / kBT;
  const uint32_t stage0 = smem_u32(sm + S::STAGE0);
  // tile t -> first row in dout / in (edge tiles start at n_kept) and its row count
  auto tile_rows = [&](int t, int64_t& row0) -> int {
    if (t < tiles_k) { row0 = int64_t(t) * kBT; return min(kBT, n_kept - t * kBT); }
    row0 = n_kept + int64_t(t - tiles_k) * kBT;
    return min(kBT, n_edge - (t - tiles_k) * kBT);
  };

  if (warp < 4 && blockIdx.x < n_tiles) {
    int64_t r0;
    const int rows = tile_rows(blockIdx.x, r0);
    prefetch_tile_rc<0>(dout + r0 * 16, in + r0 * 32, rows, stage0);
    asm volatile("cp.async.commit_group;" ::: "memory");
  }
  stage_w<32>(params, 64, sm + S::W0);
  stage_w<64>(params + 64 * 32, 16, sm + S::WO);
  if (tid == 0) {
    mbar_init(mbar, 1);
    for (int s = 0; s < F::SLOTS; s++) { mbar_init(full + s, kBT); mbar_init(empty + s, 4); }
  }
  if (warp == 0) tmem_alloc(tmem_slot, F::TMEM_COLS);
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = *tmem_slot;

  if (warp < 4) {
    // ---------------------------------------------------------------- tensor warps: mlp_bwd_rc_kernel<0>, one tile per pass
    const uint32_t tmem_row = tmem + (uint32_t(warp * 32) << 16);
    const uint32_t s_w0 = smem_u32(sm + S::W0), s_wo = smem_u32(sm + S::WO), s_h0 = smem_u32(sm + S::H0);
    constexpr uint32_t id_fwd64 = idesc_f16_f32(128, 64);
    constexpr uint32_t id_act64 = idesc_f16_f32(128, 64, 0, 1);
    constexpr uint32_t id_act32 = idesc_f16_f32(128, 32, 0, 1);
    constexpr uint32_t id_gw16 = idesc_f16_f32(64, 16, 1, 1);
    constexpr uint32_t id_gw32 = idesc_f16_f32(64, 32, 1, 1);
    uint32_t phase = 0, buf = 0;
    int it = 0, since = 0;                                       // tiles in the weight-gradient accumulators since the last flush
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, buf ^= 1, it++) {
      const int next = tile + gridDim.x;
      if (next < n_tiles) {
        int64_t r0;
        const int rows = tile_rows(next, r0);
        prefetch_tile_rc<0>(dout + r0 * 16, in + r0 * 32, rows, stage0 + (buf ^ 1) * S::STAGE_BYTES);
      }
      asm volatile("cp.async.commit_group;" ::: "memory");
      asm volatile("cp.async.wait_group 1;" ::: "memory");
      fence_async_smem();
      fence_before_sync();
      tensor_bar();
      const uint32_t sb = stage0 + buf * S::STAGE_BYTES;
      const uint32_t s_do = sb + S::DO, s_x = sb + S::X;
      const uint32_t acc = since != 0;
      // ---- F0: H0 = relu(X . W0^T)
      if (tid == 0) {
        fence_after_sync();
#pragma unroll
        for (int k = 0; k < 2; k++) mma_f16(tmem + S::C_ACT, kmajor_desc(s_x + 32 * k, 64), kmajor_desc(s_w0 + 32 * k, 64), id_fwd64, k);
        mma_commit(mbar);
      }
      mbar_wait(mbar, phase); phase ^= 1;
      fence_after_sync();
      relu_fwd_epilogue(tmem_row + S::C_ACT, sm + S::H0, tid);
      fence_before_sync();
      fence_async_smem();
      tensor_bar();
      // ---- A: dH0 = dOut . Wout ; dWout^T += H0^T . dOut
      if (tid == 0) {
        fence_after_sync();
        mma_f16(tmem + S::C_ACT, kmajor_desc(s_do, 32), mnmajor_desc(s_wo, 128, 0), id_act64, 0);
#pragma unroll
        for (int k = 0; k < 8; k++)
          mma_f16(tmem + S::C_GWO, mnmajor_desc(s_h0, 128, k), mnmajor_desc(s_do, 32, k), id_gw16, (k > 0) | acc);
        mma_commit(mbar);
      }
      mbar_wait(mbar, phase); phase ^= 1;
      fence_after_sync();
      relu_bwd_epilogue(tmem_row + S::C_ACT, sm + S::H0, sm + S::H0, tid);
      fence_before_sync();
      fence_async_smem();
      tensor_bar();
      // ---- C: dX = dH0 . W0 ; dW0 += dH0^T . X
      if (tid == 0) {
        fence_after_sync();
#pragma unroll
        for (int k = 0; k < 4; k++)
          mma_f16(tmem + S::C_ACT, kmajor_desc(s_h0 + 32 * k, 128), mnmajor_desc(s_w0, 64, k), id_act32, k);
#pragma unroll
        for (int k = 0; k < 8; k++)
          mma_f16(tmem + S::C_GW0, mnmajor_desc(s_h0, 128, k), mnmajor_desc(s_x, 64, k), id_gw32, (k > 0) | acc);
        mma_commit(mbar);
      }
      since++;
      mbar_wait(mbar, phase); phase ^= 1;
      fence_after_sync();
      // ---- dX (fp16, as f2b_mlp_bwd2 stores it) -> ring slot, word [level][row]
      const int slot = it % F::SLOTS;
      mbar_wait(empty + slot, ((it / F::SLOTS) & 1) ^ 1);        // the scatter warps are done with this slot's previous tile
      uint32_t* dst = ring + slot * F::SLOT_WORDS + tid;
#pragma unroll
      for (int q = 0; q < 2; q++) {
        uint32_t r[16];
        tmem_ld16(tmem_row + S::C_ACT + 16 * q, r);
        tmem_ld_wait();
#pragma unroll
        for (int e = 0; e < 8; e++) dst[(8 * q + e) * kBT] = pk(__uint_as_float(r[2 * e]), __uint_as_float(r[2 * e + 1]));
      }
      mbar_arrive(full + slot);
      // The UMMA's fp32 accumulation over a long chain of tiles drifts from a rounded sum: flushing after as many tiles as a CTA of
      // f2b_mlp_bwd2 accumulates keeps the weight gradient's rounding what the two-kernel sequence gives (measured: 2.6e-6
      // relative L2 apart at twice the chain length, 2e-7 between two runs of the same path).
      if (since == flush_every) { flush_field_wgrad(tmem_row, warp, lane, dparams); since = 0; }
      // the next pass's barrier orders these TMEM reads before the next tile's first MMA
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    fence_before_sync();
    tensor_bar();
    if (since) {
      fence_after_sync();
      flush_field_wgrad(tmem_row, warp, lane, dparams);
      fence_before_sync();
    }
  } else {
    // ---------------------------------------------------------------- scatter warps
    constexpr int kGroups = SCATTER_WARPS / 4;                   // warp groups taking turns over the CTA's tiles
    const int sw = warp - 4, grp = sw >> 2, quarter = sw & 3;
    int it = grp;
    for (int tile = blockIdx.x + grp * gridDim.x; tile < n_tiles; tile += kGroups * gridDim.x, it += kGroups) {
      const bool edge = tile >= tiles_k;
      const int n_seg = edge ? n_edge : n_kept;
      const int64_t i = int64_t(edge ? tile - tiles_k : tile) * kBT + quarter * 32 + lane;   // row within its segment
      const bool valid = i < n_seg;
      float x0 = 0.f, x1 = 0.f, x2 = 0.f;
      int v = -1;
      if (valid) {                                               // point + volume once for all 16 levels
        const float* p = (edge ? e_pts : pts) + i * 3;
        const float p0 = __ldg(p), p1 = __ldg(p + 1), p2 = __ldg(p + 2);
        x0 = fmul(fadd(p0, 1.f), .5f); x1 = fmul(fadd(p1, 1.f), .5f); x2 = fmul(fadd(p2, 1.f), .5f);
        v = edge ? __ldg(e_anc + i) : __ldg(anchors + i * 3);
      }
      const int slot = it % F::SLOTS;
      mbar_wait(full + slot, (it / F::SLOTS) & 1);
      const uint32_t* src = ring + slot * F::SLOT_WORDS + quarter * 32 + lane;
#pragma unroll 1
      for (int l = 0; l < F2B_N_LEVELS; l++) {                   // not unrolled: level_scale(l) stays a run-time MUFU.EX2
        const uint32_t w = src[l * kBT];
        const float2 g = __half22float2(*reinterpret_cast<const __half2*>(&w));
        hash_bwd_level(l, lane, valid, x0, x1, x2, v, g.x, g.y, prim_pool, bias_pool, n_volumes, local_size, grad_mul, grad_table);
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(empty + slot);
    }
  }
  __syncthreads();
  if (warp == 0) {
    fence_after_sync();
    tmem_dealloc(tmem, F::TMEM_COLS);
  }
}

}  // namespace f2b

using namespace f2b;

extern "C" int f2b_mlp_bwd2_tc(const void* dout_f16, const void* in_f16, const void* hidden0_f16, const void* hidden1_f16,
                               const void* params_f16, int n_hidden_matmuls, int n_pts, void* din_f16,
                               float* dparams_f32, void* stream) {
  if (n_pts <= 0) return F2B_OK;
  F2B_REQUIRE(dout_f16 && in_f16 && params_f16 && dparams_f32, "f2b_mlp_bwd: null pointer");
  F2B_REQUIRE(n_hidden_matmuls == 0 || n_hidden_matmuls == 1, "f2b_mlp_bwd: n_hidden_matmuls must be 0 or 1");
  int sms = 148;
  f2b_device_info(&sms, nullptr);
  const int n_tiles = div_up(n_pts, kBT);
  if (!hidden0_f16) {                                             // no saved activations: rebuild them on the tensor pipe
    if (n_hidden_matmuls == 0) {
      const int grid = n_tiles < sms * 4 ? n_tiles : sms * 4;     // 48 KB shared memory, 128 TMEM columns per CTA
      cudaFuncSetAttribute(mlp_bwd_rc_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, RcSmem<0>::BYTES);
      mlp_bwd_rc_kernel<0><<<grid, kBT, RcSmem<0>::BYTES, as_stream(stream)>>>((const __half*)dout_f16, (const __half*)in_f16,
                                                                              (const __half*)params_f16, n_pts, (__half*)din_f16, dparams_f32);
    } else {
      const int grid = n_tiles < sms * 2 ? n_tiles : sms * 2;     // 256 TMEM columns per CTA
      cudaFuncSetAttribute(mlp_bwd_rc_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, RcSmem<1>::BYTES);
      mlp_bwd_rc_kernel<1><<<grid, kBT, RcSmem<1>::BYTES, as_stream(stream)>>>((const __half*)dout_f16, (const __half*)in_f16,
                                                                              (const __half*)params_f16, n_pts, (__half*)din_f16, dparams_f32);
    }
    return check_launch("f2b_mlp_bwd(tcgen05, recompute)");
  }
  F2B_REQUIRE(n_hidden_matmuls == 0 || hidden1_f16, "f2b_mlp_bwd: hidden1 missing (n_hidden_matmuls == 1 with saved activations)");
  if (n_hidden_matmuls == 0) {
    const int grid = n_tiles < sms * 3 ? n_tiles : sms * 3;
    cudaFuncSetAttribute(mlp_bwd_tc_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, BwdSmem<0>::BYTES);
    mlp_bwd_tc_kernel<0><<<grid, kBT, BwdSmem<0>::BYTES, as_stream(stream)>>>(
        (const __half*)dout_f16, (const __half*)in_f16, (const __half*)hidden0_f16, (const __half*)hidden0_f16,
        (const __half*)params_f16, n_pts, (__half*)din_f16, dparams_f32);
  } else {
    const int grid = n_tiles < sms * 2 ? n_tiles : sms * 2;
    cudaFuncSetAttribute(mlp_bwd_tc_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, BwdSmem<1>::BYTES);
    mlp_bwd_tc_kernel<1><<<grid, kBT, BwdSmem<1>::BYTES, as_stream(stream)>>>(
        (const __half*)dout_f16, (const __half*)in_f16, (const __half*)hidden0_f16, (const __half*)hidden1_f16,
        (const __half*)params_f16, n_pts, (__half*)din_f16, dparams_f32);
  }
  return check_launch("f2b_mlp_bwd(tcgen05)");
}

extern "C" int f2b_mlp_bwd_tc(const void* dout_f16, const void* in_f16, const void* hidden_save_f16,
                              const void* params_f16, int n_hidden_matmuls, int n_pts, void* din_f16,
                              float* dparams_f32, void* stream) {
  if (n_pts <= 0) return F2B_OK;
  F2B_REQUIRE(hidden_save_f16, "f2b_mlp_bwd: null pointer");
  const __half* h = (const __half*)hidden_save_f16;
  return f2b_mlp_bwd2_tc(dout_f16, in_f16, h, h + size_t(n_hidden_matmuls ? 1 : 0) * n_pts * 64, params_f16, n_hidden_matmuls, n_pts,
                         din_f16, dparams_f32, stream);
}

template <int SW, int CTAS>
static int launch_field_bwd_scatter(int grid, int flush_every, const void* dout_f16, const void* in_f16, const void* params_f16, int n_kept,
                                    const float* pts, const int* anchors, int n_edge, const float* e_pts, const int* e_anc,
                                    const int* prim_pool, const float* bias_pool, int n_volumes, int local_size, float grad_mul,
                                    float* dparams_f32, float* grad_table, cudaStream_t st) {
  cudaFuncSetAttribute(field_bwd_scatter_kernel<SW, CTAS>, cudaFuncAttributeMaxDynamicSharedMemorySize, FbsSmem<SW>::BYTES);
  field_bwd_scatter_kernel<SW, CTAS><<<grid, kBT + 32 * SW, FbsSmem<SW>::BYTES, st>>>(
      (const __half*)dout_f16, (const __half*)in_f16, (const __half*)params_f16, n_kept, pts, anchors, n_edge, e_pts, e_anc, prim_pool,
      bias_pool, n_volumes, local_size, grad_mul, dparams_f32, grad_table, flush_every);
  return check_launch("f2b_field_bwd_scatter");
}

extern "C" int f2b_field_bwd_scatter(const void* dout_f16, const void* in_f16, const void* params_f16, int n_kept, const float* pts,
                                     const int* anchors, int n_edge, const float* e_pts, const int* e_anc, const int* prim_pool,
                                     const float* bias_pool, int n_volumes, int local_size, float grad_mul, float* dparams_f32,
                                     float* grad_table, void* stream) {
  F2B_REQUIRE(n_kept >= 0 && n_edge >= 0, "f2b_field_bwd_scatter: negative row count");
  if (n_kept + n_edge <= 0) return F2B_OK;
  F2B_REQUIRE(dout_f16 && in_f16 && params_f16 && prim_pool && bias_pool && dparams_f32 && grad_table,
              "f2b_field_bwd_scatter: null pointer");
  F2B_REQUIRE((n_kept == 0 || (pts && anchors)) && (n_edge == 0 || (e_pts && e_anc)), "f2b_field_bwd_scatter: null point segment");
  F2B_REQUIRE(n_volumes > 0 && local_size > 0 && (local_size % 2) == 0, "f2b_field_bwd_scatter: bad n_volumes/local_size");
  // scatter warps per CTA x resident CTAs per SM: default 8 x 2, the fastest of the sweep {4, 8} x {2, 3} + 12 x 2 on B200
  // (profiles/r03a_sweep.jsonl, profiles/r03b_sweep.jsonl); F2B_FBS_WARPS / F2B_FBS_CTAS select another point of it
  static int warps = -1, ctas = -1;
  if (warps < 0) {
    const char* w = getenv("F2B_FBS_WARPS");
    const char* c = getenv("F2B_FBS_CTAS");
    warps = w ? atoi(w) : 8;
    ctas = c ? atoi(c) : 2;
    if (warps != 4 && warps != 12) warps = 8;
    if (ctas != 3) ctas = 2;
  }
  int sms = 148;
  f2b_device_info(&sms, nullptr);
  const int n_tiles = div_up(n_kept, kBT) + div_up(n_edge, kBT);
  const int grid = n_tiles < sms * ctas ? n_tiles : sms * ctas;
  const cudaStream_t st = as_stream(stream);
  // weight-gradient chain per flush: the tiles one CTA of f2b_mlp_bwd2 (4 CTAs per SM) accumulates before its single flush
  const int flush_every = div_up(n_tiles, int64_t(sms) * 4);
#define F2B_FBS(SW, CT) launch_field_bwd_scatter<SW, CT>(grid, flush_every, dout_f16, in_f16, params_f16, n_kept, pts, anchors, n_edge, e_pts, e_anc, \
                                                         prim_pool, bias_pool, n_volumes, local_size, grad_mul, dparams_f32, grad_table, st)
  if (warps == 12) return F2B_FBS(12, 2);                           // 12 x 3 would spill at 40 registers
  if (warps == 8) return ctas == 2 ? F2B_FBS(8, 2) : F2B_FBS(8, 3);
  return ctas == 2 ? F2B_FBS(4, 2) : F2B_FBS(4, 3);
#undef F2B_FBS
}
