// Attention backward with the gated relative-position bias (autograd of WavLM/modules.py:521-563), tcgen05 + TMEM + TMA.
//
// Two tensor-core kernels, each recomputing P from the saved log-sum-exp (flash-attention style), so that every
// reduction is either a TMEM accumulation or thread-local:
//   * dK/dV kernel: CTA = 128 keys of one (b,h), loops over query tiles.  Works in the TRANSPOSED orientation
//       S^T = K Q^T, dP^T = V dO^T  (thread = key row), writes P^T and dS^T once to shared memory (K-major operand
//       layout) and accumulates dV += P^T dO, dK += dS^T Q in TMEM across the whole loop.
//   * dQ kernel: CTA = 128 queries, loops over key tiles (thread = query row): dQ += dS K accumulates in TMEM;
//       d gate[b,h,i] = sum_j dS_ij tab[j-i] is a thread-local row sum;  d tab[h,delta] = sum_{b,i} gate_i dS_{i,i+delta}
//       is a diagonal sum: the tile gate_i*dS is staged in shared memory (bf16) and re-read along diagonals, one diagonal
//       pair per thread, then accumulated per CTA and flushed with atomics (the table is shared by all layers, SURVEY S10).
//   dS = P o (dP - Delta), Delta_i = sum_d dO_id O_id (small pre-kernel).
#include "../../include/unispeech_b200.h"
#include "attn_common.cuh"
#include "common.h"

namespace b200 {

__device__ __forceinline__ float fast_exp2_b(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// ------------------------------------------------------------------------------------------------ Delta
__global__ void __launch_bounds__(256) attn_delta_kernel(const __nv_bfloat16* __restrict__ o,
                                                         const __nv_bfloat16* __restrict__ dout, int B, int T, int H,
                                                         float* __restrict__ delta) {
  pdl_grid_sync();
  // one warp per (b,t): lane handles 2 columns of each head
  const int lane = threadIdx.x & 31;
  const long long row = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  if (row >= static_cast<long long>(B) * T) return;
  const int D = H * kHeadDim;
  const long long b = row / T, t = row % T;
  for (int h = 0; h < H; ++h) {
    const float2 a = unpack_bf16x2(*reinterpret_cast<const uint32_t*>(o + row * D + h * kHeadDim + lane * 2));
    const float2 g = unpack_bf16x2(*reinterpret_cast<const uint32_t*>(dout + row * D + h * kHeadDim + lane * 2));
    const float s = warp_sum(a.x * g.x + a.y * g.y);
    if (lane == 0) delta[(b * H + h) * T + t] = s;
  }
}

// ------------------------------------------------------------------------------------------------ dK / dV
constexpr int kKvK = 0, kKvV = 16384, kKvQ = 32768, kKvDO = 65536, kKvPT = 98304, kKvDST = 131072, kKvVec = 163840,
              kKvTab = 167936;

template <bool HAS_BIAS>
__global__ void __launch_bounds__(256, 1) attn_bwd_dkv_kernel(const __grid_constant__ CUtensorMap tm_qkv,
                                                              const __grid_constant__ CUtensorMap tm_do,
                                                              const __grid_constant__ AttnParams p) {
  pdl_grid_sync();
  const int tid = threadIdx.x, warp = tid >> 5;
  const int k0 = blockIdx.x * kAttnTile, h = blockIdx.y, b = blockIdx.z;
  const int T = p.T, D = p.D, N = p.n_tiles;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);  // 1024-aligned, still a __shared__ pointer (LDS/STS, not generic)
  uint8_t* sK = smem + kKvK;
  uint8_t* sV = smem + kKvV;
  uint8_t* sQ = smem + kKvQ;    // 2 stages
  uint8_t* sDO = smem + kKvDO;  // 2 stages
  uint8_t* sPT = smem + kKvPT;
  uint8_t* sDST = smem + kKvDST;
  float4* colvec = reinterpret_cast<float4*>(smem + kKvVec);  // [2][128] {lse2, delta, gate*log2e, unused}
  float* tab_s = reinterpret_cast<float*>(smem + kKvTab);     // [(N+1)*128]

  __shared__ uint64_t kv_full, qdo_full[2], st_full, acc_done;
  __shared__ uint32_t tmem_base_s;

  if (tid == 0) {
    tma_prefetch_desc(&tm_qkv);
    tma_prefetch_desc(&tm_do);
    mbar_init(&kv_full, 1);
    mbar_init(&qdo_full[0], 1);
    mbar_init(&qdo_full[1], 1);
    mbar_init(&st_full, 1);
    mbar_init(&acc_done, 1);
    fence_mbar_init();
  }
  __syncwarp();
  if (warp == 0) tmem_alloc(&tmem_base_s, 512);

  // bias table slice for this key tile: tab_s[l] = tab[h, l + base], base = k0 - (N*128-1) + T-1; element (r, i) -> l = r + N*128-1 - i
  if (HAS_BIAS) {
    const int len = (N + 1) * kAttnTile;
    const int base = k0 - (N * kAttnTile - 1) + (T - 1);
    for (int l = tid; l < len; l += blockDim.x) {
      const int gi = l + base;
      tab_s[l] = (gi >= 0 && gi < 2 * T - 1) ? p.tab[static_cast<long long>(h) * (2 * T - 1) + gi] : 0.f;
    }
  }
  auto load_colvec = [&](int qi) {
    if (tid >= kAttnTile) return;  // one loader per query column
    const int i = qi * kAttnTile + tid;
    float4 v;
    if (i < T) {
      const long long idx = (static_cast<long long>(b) * p.H + h) * T + i;
      v.x = p.lse[idx];
      v.y = p.delta[idx];
      v.z = (HAS_BIAS ? ((p.gate != nullptr) ? p.gate[idx] : 1.0f) : 0.f) * kLog2e;
    } else {
      v.x = INFINITY;  // p = exp2(-inf) = 0 for out-of-range queries
      v.y = 0.f;
      v.z = 0.f;
    }
    v.w = 0.f;
    colvec[(qi & 1) * kAttnTile + tid] = v;
  };
  load_colvec(0);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;
  constexpr uint32_t idesc_s = make_idesc_bf16(128, 128, 0, 0);
  constexpr uint32_t idesc_acc = make_idesc_bf16(128, 64, 0, 1);

  auto load_qdo = [&](int qi) {
    const int s = qi & 1;
    mbar_expect_tx(&qdo_full[s], 32768);
    tma_load_4d(sQ + s * 16384, &tm_qkv, &qdo_full[s], h * kHeadDim, qi * kAttnTile, b, 0);
    tma_load_4d(sDO + s * 16384, &tm_do, &qdo_full[s], h * kHeadDim, qi * kAttnTile, b, 0);
  };
  auto issue_st = [&](int qi) {  // S^T = K Q^T -> cols [0,128);  dP^T = V dO^T -> cols [128,256)
    const int s = qi & 1;
    const uint32_t ak = smem_u32(sK), av = smem_u32(sV), bq = smem_u32(sQ + s * 16384), bd = smem_u32(sDO + s * 16384);
#pragma unroll
    for (int k = 0; k < 4; ++k)
      umma_bf16(tmem, make_smem_desc_sw128(ak + k * 32, 16, 1024), make_smem_desc_sw128(bq + k * 32, 16, 1024), idesc_s,
                k > 0 ? 1u : 0u);
#pragma unroll
    for (int k = 0; k < 4; ++k)
      umma_bf16(tmem + 128, make_smem_desc_sw128(av + k * 32, 16, 1024), make_smem_desc_sw128(bd + k * 32, 16, 1024),
                idesc_s, k > 0 ? 1u : 0u);
    umma_commit(&st_full);
  };

  if (tid == 0) {
    mbar_expect_tx(&kv_full, 32768);
    tma_load_4d(sK, &tm_qkv, &kv_full, D + h * kHeadDim, k0, b, 0);
    tma_load_4d(sV, &tm_qkv, &kv_full, 2 * D + h * kHeadDim, k0, b, 0);
    load_qdo(0);
    if (N > 1) load_qdo(1);
    mbar_wait(&kv_full, 0);
    mbar_wait(&qdo_full[0], 0);
    tc_fence_after();
    issue_st(0);
  }
  __syncwarp();

  // two threads per key row: warpgroup `half` handles query columns [64*half, 64*half+64) of every tile (two warps per
  // scheduler hide the latency of this issue-bound phase; the MMAs, TMEM and shared-memory layout are unchanged)
  const int r = tid & (kAttnTile - 1);  // key row inside the tile
  const int half = tid >> 7;
  const int key = k0 + r;
  const bool key_valid = key < T;
  const bool key_masked = !key_valid || (p.key_pad != nullptr && p.key_pad[static_cast<long long>(b) * T + key] != 0);
  const float kb = key_masked ? -INFINITY : 0.f;
  const float sc = p.scale * kLog2e;
  const float* tabrow = tab_s + r + N * kAttnTile - 1;
  const uint32_t lane_addr = static_cast<uint32_t>((warp & 3) * 32) << 16;

  for (int qi = 0; qi < N; ++qi) {
    const int st = qi & 1;
    const int i0 = qi * kAttnTile;
    mbar_wait(&st_full, qi & 1);
    tc_fence_after();
    // st_full(qi) was committed after the dV/dK MMAs of tile qi-1: their operands (PT/dST, Q/dO stage st^1) are free now
    if (tid == 0 && qi >= 1 && qi + 1 < N) load_qdo(qi + 1);
    __syncwarp();
    const float4* cv = colvec + st * kAttnTile;
#pragma unroll 1
    for (int c0 = half * 64; c0 < half * 64 + 64; c0 += 32) {
      uint32_t su[32], du[32];
      tmem_ld_32x32b_x32(tmem + lane_addr + c0, su);
      tmem_ld_32x32b_x32(tmem + lane_addr + 128 + c0, du);
      tmem_ld_wait();
      float pv[32], dv[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        const float4 c = cv[c0 + j];
        float x = __uint_as_float(su[j]) * sc + kb;
        if (HAS_BIAS) x = fmaf(c.z, tabrow[-(i0 + c0 + j)], x);
        const float pr = fast_exp2_b(x - c.x);
        pv[j] = pr;
        dv[j] = pr * (__uint_as_float(du[j]) - c.y) * p.scale;
      }
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        uint4 w;
        w.x = pack_bf16x2(pv[g * 8 + 0], pv[g * 8 + 1]);
        w.y = pack_bf16x2(pv[g * 8 + 2], pv[g * 8 + 3]);
        w.z = pack_bf16x2(pv[g * 8 + 4], pv[g * 8 + 5]);
        w.w = pack_bf16x2(pv[g * 8 + 6], pv[g * 8 + 7]);
        store_sw128_chunk(sPT, r, (c0 >> 3) + g, w);
        w.x = pack_bf16x2(dv[g * 8 + 0], dv[g * 8 + 1]);
        w.y = pack_bf16x2(dv[g * 8 + 2], dv[g * 8 + 3]);
        w.z = pack_bf16x2(dv[g * 8 + 4], dv[g * 8 + 5]);
        w.w = pack_bf16x2(dv[g * 8 + 6], dv[g * 8 + 7]);
        store_sw128_chunk(sDST, r, (c0 >> 3) + g, w);
      }
    }
    if (qi + 1 < N) load_colvec(qi + 1);
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    if (tid == 0) {
      tc_fence_after();
      const uint32_t apt = smem_u32(sPT), ads = smem_u32(sDST), bdo = smem_u32(sDO + st * 16384),
                     bq = smem_u32(sQ + st * 16384);
#pragma unroll
      for (int k = 0; k < 8; ++k) {  // dV += P^T dO ; dK += dS^T Q   (K = 128 queries, B operands MN-major)
        const uint32_t aoff = (k >> 2) * 16384 + (k & 3) * 32;
        umma_bf16(tmem + 256, make_smem_desc_sw128(apt + aoff, 16, 1024), make_smem_desc_sw128(bdo + k * 2048, 8192, 1024),
                  idesc_acc, (qi > 0 || k > 0) ? 1u : 0u);
      }
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const uint32_t aoff = (k >> 2) * 16384 + (k & 3) * 32;
        umma_bf16(tmem + 320, make_smem_desc_sw128(ads + aoff, 16, 1024), make_smem_desc_sw128(bq + k * 2048, 8192, 1024),
                  idesc_acc, (qi > 0 || k > 0) ? 1u : 0u);
      }
      if (qi + 1 < N) {
        mbar_wait(&qdo_full[st ^ 1], ((qi + 1) >> 1) & 1);
        tc_fence_after();
        issue_st(qi + 1);
      } else {
        umma_commit(&acc_done);
      }
    }
    __syncwarp();
  }
  mbar_wait(&acc_done, 0);
  tc_fence_after();

  {
    uint32_t t0[32], t1[32];
#pragma unroll 1
    for (int which = half; which <= half; ++which) {  // warpgroup 0 writes dV (cols 256..), warpgroup 1 dK (cols 320..)
      const uint32_t col = 256 + which * 64;
      tmem_ld_32x32b_x32(tmem + lane_addr + col, t0);
      tmem_ld_32x32b_x32(tmem + lane_addr + col + 32, t1);
      tmem_ld_wait();
      if (key_valid) {
        __nv_bfloat16* dst = p.dqkv + (static_cast<long long>(b) * T + key) * (3 * D) + (which == 0 ? 2 * D : D) +
                             h * kHeadDim;
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          uint4 w;
          w.x = pack_bf16x2(__uint_as_float(t0[g * 8 + 0]), __uint_as_float(t0[g * 8 + 1]));
          w.y = pack_bf16x2(__uint_as_float(t0[g * 8 + 2]), __uint_as_float(t0[g * 8 + 3]));
          w.z = pack_bf16x2(__uint_as_float(t0[g * 8 + 4]), __uint_as_float(t0[g * 8 + 5]));
          w.w = pack_bf16x2(__uint_as_float(t0[g * 8 + 6]), __uint_as_float(t0[g * 8 + 7]));
          *reinterpret_cast<uint4*>(dst + g * 8) = w;
          w.x = pack_bf16x2(__uint_as_float(t1[g * 8 + 0]), __uint_as_float(t1[g * 8 + 1]));
          w.y = pack_bf16x2(__uint_as_float(t1[g * 8 + 2]), __uint_as_float(t1[g * 8 + 3]));
          w.z = pack_bf16x2(__uint_as_float(t1[g * 8 + 4]), __uint_as_float(t1[g * 8 + 5]));
          w.w = pack_bf16x2(__uint_as_float(t1[g * 8 + 6]), __uint_as_float(t1[g * 8 + 7]));
          *reinterpret_cast<uint4*>(dst + 32 + g * 8) = w;
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    __syncwarp();
    tmem_dealloc(tmem, 512);
  }
}

// ------------------------------------------------------------------------------------------------ dQ / d gate / d tab
constexpr int kDqQ = 0, kDqDO = 16384, kDqK = 32768, kDqV = 65536, kDqDS = 98304, kDqW = 131072;
constexpr int kWStride = 130;  // bf16 elements per staged row (65 words: conflict-free row writes and diagonal reads)
constexpr int kDqTab = kDqW + 128 * kWStride * 2 + 64;  // 164416, 16B aligned

template <bool HAS_BIAS>
__global__ void __launch_bounds__(256, 1) attn_bwd_dq_kernel(const __grid_constant__ CUtensorMap tm_qkv,
                                                             const __grid_constant__ CUtensorMap tm_do,
                                                             const __grid_constant__ AttnParams p) {
  pdl_grid_sync();
  const int tid = threadIdx.x, warp = tid >> 5;
  const int q0 = blockIdx.x * kAttnTile, h = blockIdx.y, b = blockIdx.z;
  const int T = p.T, D = p.D, N = p.n_tiles;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);  // 1024-aligned, still a __shared__ pointer (LDS/STS, not generic)
  uint8_t* sQ = smem + kDqQ;
  uint8_t* sDO = smem + kDqDO;
  uint8_t* sK = smem + kDqK;  // 2 stages
  uint8_t* sV = smem + kDqV;  // 2 stages
  uint8_t* sDS = smem + kDqDS;
  __nv_bfloat16* sW = reinterpret_cast<__nv_bfloat16*>(smem + kDqW);
  float* tab_s = reinterpret_cast<float*>(smem + kDqTab);
  float* kbias = tab_s + (N + 1) * kAttnTile;
  float* dtab_acc = kbias + N * kAttnTile;  // [(N+1)*128]
  int* tile_flags = reinterpret_cast<int*>(dtab_acc + (N + 1) * kAttnTile);

  __shared__ uint64_t qdo_full, kv_full[2], s_full, acc_done;
  __shared__ uint32_t tmem_base_s;

  if (tid == 0) {
    tma_prefetch_desc(&tm_qkv);
    tma_prefetch_desc(&tm_do);
    mbar_init(&qdo_full, 1);
    mbar_init(&kv_full[0], 1);
    mbar_init(&kv_full[1], 1);
    mbar_init(&s_full, 1);
    mbar_init(&acc_done, 1);
    fence_mbar_init();
  }
  __syncwarp();
  if (warp == 0) tmem_alloc(&tmem_base_s, 512);
  if (HAS_BIAS) {
    load_tab_slice(tab_s, p.tab, h, T, q0, N);
    for (int i = tid; i < (N + 1) * kAttnTile; i += blockDim.x) dtab_acc[i] = 0.f;
  }
  load_key_mask(kbias, tile_flags, p.key_pad, b, T, N);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;
  constexpr uint32_t idesc_s = make_idesc_bf16(128, 128, 0, 0);
  constexpr uint32_t idesc_acc = make_idesc_bf16(128, 64, 0, 1);

  auto load_kv = [&](int n) {
    const int s = n & 1;
    mbar_expect_tx(&kv_full[s], 32768);
    tma_load_4d(sK + s * 16384, &tm_qkv, &kv_full[s], D + h * kHeadDim, n * kAttnTile, b, 0);
    tma_load_4d(sV + s * 16384, &tm_qkv, &kv_full[s], 2 * D + h * kHeadDim, n * kAttnTile, b, 0);
  };
  auto issue_s = [&](int n) {  // S = Q K^T -> cols [0,128);  dP = dO V^T -> cols [128,256)
    const int s = n & 1;
    const uint32_t aq = smem_u32(sQ), ad = smem_u32(sDO), bk = smem_u32(sK + s * 16384), bv = smem_u32(sV + s * 16384);
#pragma unroll
    for (int k = 0; k < 4; ++k)
      umma_bf16(tmem, make_smem_desc_sw128(aq + k * 32, 16, 1024), make_smem_desc_sw128(bk + k * 32, 16, 1024), idesc_s,
                k > 0 ? 1u : 0u);
#pragma unroll
    for (int k = 0; k < 4; ++k)
      umma_bf16(tmem + 128, make_smem_desc_sw128(ad + k * 32, 16, 1024), make_smem_desc_sw128(bv + k * 32, 16, 1024),
                idesc_s, k > 0 ? 1u : 0u);
    umma_commit(&s_full);
  };

  if (tid == 0) {
    mbar_expect_tx(&qdo_full, 32768);
    tma_load_4d(sQ, &tm_qkv, &qdo_full, h * kHeadDim, q0, b, 0);
    tma_load_4d(sDO, &tm_do, &qdo_full, h * kHeadDim, q0, b, 0);
    load_kv(0);
    if (N > 1) load_kv(1);
    mbar_wait(&qdo_full, 0);
    mbar_wait(&kv_full[0], 0);
    tc_fence_after();
    issue_s(0);
  }
  __syncwarp();

  const int r = tid & (kAttnTile - 1);  // two threads per query row, see the dK/dV kernel
  const int half = tid >> 7;
  const bool row_valid = (q0 + r) < T;
  const long long ridx = (static_cast<long long>(b) * p.H + h) * T + q0 + r;
  const float lse2 = row_valid ? p.lse[ridx] : INFINITY;
  const float delta = row_valid ? p.delta[ridx] : 0.f;
  float g = 0.f;
  if (HAS_BIAS) g = (p.gate != nullptr && row_valid) ? p.gate[ridx] : (row_valid ? 1.0f : 0.f);
  const float gl = g * kLog2e;
  const float sc = p.scale * kLog2e;
  const float* tabrow = tab_s + (kAttnTile - 1 - r);
  const uint32_t lane_addr = static_cast<uint32_t>((warp & 3) * 32) << 16;
  float dgate_acc = 0.f;
  uint32_t* wrow = reinterpret_cast<uint32_t*>(sW) + r * (kWStride / 2);

  for (int n = 0; n < N; ++n) {
    const int st = n & 1;
    const int k0 = n * kAttnTile;
    mbar_wait(&s_full, n & 1);
    tc_fence_after();
    // s_full(n) was committed after the dQ MMA of tile n-1: dS smem and K/V stage st^1 are free now
    if (tid == 0 && n >= 1 && n + 1 < N) load_kv(n + 1);
    __syncwarp();
    const bool msk = tile_flags[n] != 0;
#pragma unroll 1
    for (int c0 = half * 64; c0 < half * 64 + 64; c0 += 32) {
      uint32_t su[32], du[32];
      tmem_ld_32x32b_x32(tmem + lane_addr + c0, su);
      tmem_ld_32x32b_x32(tmem + lane_addr + 128 + c0, du);
      tmem_ld_wait();
      float dsv[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        float x = __uint_as_float(su[j]) * sc;
        float tb = 0.f;
        if (HAS_BIAS) {
          tb = tabrow[k0 + c0 + j];
          x = fmaf(gl, tb, x);
        }
        if (msk) x += kbias[k0 + c0 + j];
        const float pr = fast_exp2_b(x - lse2);
        const float ds = pr * (__uint_as_float(du[j]) - delta);
        if (HAS_BIAS) dgate_acc = fmaf(ds, tb, dgate_acc);
        dsv[j] = ds;
      }
#pragma unroll
      for (int gq = 0; gq < 4; ++gq) {
        uint4 w;
        w.x = pack_bf16x2(dsv[gq * 8 + 0] * p.scale, dsv[gq * 8 + 1] * p.scale);
        w.y = pack_bf16x2(dsv[gq * 8 + 2] * p.scale, dsv[gq * 8 + 3] * p.scale);
        w.z = pack_bf16x2(dsv[gq * 8 + 4] * p.scale, dsv[gq * 8 + 5] * p.scale);
        w.w = pack_bf16x2(dsv[gq * 8 + 6] * p.scale, dsv[gq * 8 + 7] * p.scale);
        store_sw128_chunk(sDS, r, (c0 >> 3) + gq, w);
      }
      if (HAS_BIAS) {
#pragma unroll
        for (int j = 0; j < 16; ++j) wrow[(c0 >> 1) + j] = pack_bf16x2(g * dsv[2 * j], g * dsv[2 * j + 1]);
      }
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    if (tid == 0) {
      tc_fence_after();
      const uint32_t ads = smem_u32(sDS), bk = smem_u32(sK + st * 16384);
#pragma unroll
      for (int k = 0; k < 8; ++k) {  // dQ += dS K   (K = 128 keys, B operand MN-major)
        const uint32_t aoff = (k >> 2) * 16384 + (k & 3) * 32;
        umma_bf16(tmem + 256, make_smem_desc_sw128(ads + aoff, 16, 1024), make_smem_desc_sw128(bk + k * 2048, 8192, 1024),
                  idesc_acc, (n > 0 || k > 0) ? 1u : 0u);
      }
      if (n + 1 < N) {
        mbar_wait(&kv_full[st ^ 1], ((n + 1) >> 1) & 1);
        tc_fence_after();
        issue_s(n + 1);
      } else {
        umma_commit(&acc_done);
      }
    }
    __syncwarp();
    if (HAS_BIAS) {
      // diagonal sums of the staged tile: thread d sums W[rr][(rr+d) & 127]; columns wrap once, giving two diagonals
      const int d = r;
      float acc_pos = 0.f, acc_neg = 0.f;
#pragma unroll 8
      for (int rr = half * 64; rr < half * 64 + 64; ++rr) {
        const int c = (rr + d) & (kAttnTile - 1);
        const float v = __bfloat162float(sW[rr * kWStride + c]);
        if (rr + d < kAttnTile) acc_pos += v; else acc_neg += v;
      }
      atomicAdd(&dtab_acc[k0 + d + kAttnTile - 1], acc_pos);
      if (d > 0) atomicAdd(&dtab_acc[k0 + d - 1], acc_neg);
      __syncthreads();  // sW is rewritten by the next tile
    }
  }
  mbar_wait(&acc_done, 0);
  tc_fence_after();
  {
    uint32_t t0[32];
    tmem_ld_32x32b_x32(tmem + lane_addr + 256 + half * 32, t0);  // each warpgroup writes 32 of the 64 dQ columns
    tmem_ld_wait();
    __shared__ float dgate_x[kAttnTile];
    if (HAS_BIAS && half == 1) dgate_x[r] = dgate_acc;
    __syncthreads();
    if (HAS_BIAS && half == 0) dgate_acc += dgate_x[r];
    if (row_valid) {
      __nv_bfloat16* dst = p.dqkv + (static_cast<long long>(b) * T + q0 + r) * (3 * D) + h * kHeadDim + half * 32;
#pragma unroll
      for (int gq = 0; gq < 4; ++gq) {
        uint4 w;
        w.x = pack_bf16x2(__uint_as_float(t0[gq * 8 + 0]), __uint_as_float(t0[gq * 8 + 1]));
        w.y = pack_bf16x2(__uint_as_float(t0[gq * 8 + 2]), __uint_as_float(t0[gq * 8 + 3]));
        w.z = pack_bf16x2(__uint_as_float(t0[gq * 8 + 4]), __uint_as_float(t0[gq * 8 + 5]));
        w.w = pack_bf16x2(__uint_as_float(t0[gq * 8 + 6]), __uint_as_float(t0[gq * 8 + 7]));
        *reinterpret_cast<uint4*>(dst + gq * 8) = w;
      }
      if (HAS_BIAS && half == 0 && p.dgate != nullptr) p.dgate[ridx] = dgate_acc;
    }
  }
  if (HAS_BIAS && p.dtab != nullptr) {
    __syncthreads();
    const int base = (T - 1) - (q0 + kAttnTile - 1);
    for (int i = tid; i < (N + 1) * kAttnTile; i += blockDim.x) {
      const int gi = i + base;
      const float v = dtab_acc[i];
      if (gi >= 0 && gi < 2 * T - 1 && v != 0.f) atomicAdd(p.dtab + static_cast<long long>(h) * (2 * T - 1) + gi, v);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    __syncwarp();
    tmem_dealloc(tmem, 512);
  }
}

int make_qkv_tmap(CUtensorMap* out, const void* qkv, int T, int B, int D3, int box_rows);

// Delta = rowsum(dO * O) for the long-utterance backward (attn_long.cu)
cudaError_t launch_attn_delta(const void* out, const void* dout, int B, int T, int H, float* delta, cudaStream_t st) {
  const long long rows = static_cast<long long>(B) * T;
  return launch_pdl(attn_delta_kernel, dim3(static_cast<unsigned>(ceil_div_ll(rows * 32, 256))), dim3(256), 0, st,
                    static_cast<const __nv_bfloat16*>(out), static_cast<const __nv_bfloat16*>(dout), B, T, H, delta);
}

}  // namespace b200

using namespace b200;

extern "C" {

// Backward of b200s_attn_fwd.  out/dout: bf16 [B,T,D]; lse from the forward; delta: fp32 [B,H,T] workspace;
// dqkv: bf16 [B,T,3D] (fully written for valid rows); dgate: fp32 [B,H,T] (written); dtab: fp32 [H,2T-1] (ACCUMULATED with
// atomics -- the caller zeroes it once per step, the table is shared by all layers).  gate/tab/dgate/dtab NULL = no bias.
int b200s_attn_bwd(const void* qkv, const void* out, const void* dout, const float* gate, const float* tab,
                   const uint8_t* key_pad, const float* lse, float* delta, void* dqkv, float* dgate, float* dtab, int B,
                   int T, int H, float scale, b200s_stream stream) {
  B200_CHECK_ARG(qkv && out && dout && lse && delta && dqkv, "attn_bwd: null pointer");
  B200_CHECK_ARG(T >= 1 && T <= 4096, "attn_bwd: T=%d out of range (1..4096)", T);
  B200_CHECK_ARG(!tab || (dgate && dtab), "attn_bwd: bias given but dgate/dtab missing");
  const int D = H * kHeadDim;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long rows = static_cast<long long>(B) * T;
  B200_CHECK_CUDA(launch_pdl(attn_delta_kernel, dim3(static_cast<unsigned>(ceil_div_ll(rows * 32, 256))), dim3(256), 0, st, 
      static_cast<const __nv_bfloat16*>(out), static_cast<const __nv_bfloat16*>(dout), B, T, H, delta));
  B200_CHECK_LAUNCH();

  CUtensorMap tm_qkv, tm_do;
  if (make_qkv_tmap(&tm_qkv, qkv, T, B, 3 * D, kAttnTile)) return -3;
  if (make_qkv_tmap(&tm_do, dout, T, B, D, kAttnTile)) return -3;
  AttnParams p;
  memset(&p, 0, sizeof(p));
  p.T = T; p.H = H; p.B = B; p.D = D;
  p.n_tiles = ceil_div(T, kAttnTile);
  p.scale = scale;
  p.gate = gate; p.tab = tab; p.key_pad = key_pad;
  p.lse = const_cast<float*>(lse);
  p.dout = static_cast<const __nv_bfloat16*>(dout);
  p.delta = delta;
  p.dqkv = static_cast<__nv_bfloat16*>(dqkv);
  p.dgate = dgate;
  p.dtab = dtab;
  dim3 grid(p.n_tiles, H, B);
  const int N = p.n_tiles;
  const int smem_kv = kKvTab + sizeof(float) * (N + 1) * kAttnTile + 1024;
  const int smem_dq = kDqTab + sizeof(float) * ((N + 1) * kAttnTile * 2 + N * kAttnTile) + sizeof(int) * N + 1024;
  if (tab != nullptr) {
    B200_CHECK_CUDA(cudaFuncSetAttribute(attn_bwd_dkv_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_kv));
    B200_CHECK_CUDA(launch_pdl(attn_bwd_dkv_kernel<true>, dim3(grid), dim3(256), smem_kv, st, tm_qkv, tm_do, p));
    B200_CHECK_LAUNCH();
    B200_CHECK_CUDA(cudaFuncSetAttribute(attn_bwd_dq_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_dq));
    B200_CHECK_CUDA(launch_pdl(attn_bwd_dq_kernel<true>, dim3(grid), dim3(256), smem_dq, st, tm_qkv, tm_do, p));
  } else {
    B200_CHECK_CUDA(cudaFuncSetAttribute(attn_bwd_dkv_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_kv));
    B200_CHECK_CUDA(launch_pdl(attn_bwd_dkv_kernel<false>, dim3(grid), dim3(256), smem_kv, st, tm_qkv, tm_do, p));
    B200_CHECK_LAUNCH();
    B200_CHECK_CUDA(cudaFuncSetAttribute(attn_bwd_dq_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_dq));
    B200_CHECK_CUDA(launch_pdl(attn_bwd_dq_kernel<false>, dim3(grid), dim3(256), smem_dq, st, tm_qkv, tm_do, p));
  }
  B200_CHECK_LAUNCH();
  return 0;
}

}  // extern "C"
