// Attention forward and backward for long utterances (up to 16384 frames), tcgen05 + TMEM + TMA (sm_100a).
//
// Same math, operands and outputs as attn_fwd.cu / attn_bwd.cu; see those files for the pipeline.  What differs is that no
// shared-memory array grows with T: attn_fwd.cu keeps the CTA's whole slice of the bias table and the whole key mask, which
// limits it to T <= 3072 with the bias, and attn_bwd.cu keeps table, mask and d-table slices, which limits it to T <= 4096.
// Here every key (or query) tile stages just the window it needs:
//   * forward: per key tile, the 128 + 256 - 1 table entries its 256 query rows read (four shifted copies, as in attn_fwd.cu)
//     and the tile's 128 key-mask values, filled by the TMA warp into a two-stage ring beside K / V;
//   * backward: per tile, the 255-entry table window and (dQ kernel) the tile's key mask, double-buffered and filled by the
//     CTA's threads in the slot before the barrier that already separates two tiles; d tab is accumulated per tile window and
//     flushed with atomics.
// Saturated bias.  The WavLM bucket of a relative distance delta is constant for |delta| >= R (the log branch of the bucketing
// clamps to its last bucket), so tab[h, delta] = tab[h, sign(delta) R] there.  The caller passes R (`tab_radius`; R = T - 1 is
// always exact).  A tile whose every (query, key) pair has |delta| >= R on one side ("off band") adds the per-row constant
// gate_i * tab[h, +-R]: the forward skips the table window, and the backward sums that tile's gate_i * dS_ij into two scalars
// added to d tab at delta = +-R instead of diagonal by diagonal.
#include "../../include/unispeech_b200.h"
#include "attn_common.cuh"
#include "common.h"
#include <type_traits>

namespace b200 {

__device__ __forceinline__ float fast_exp2_l(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ void mbar_arrive_rel_l(uint64_t* bar) {
  asm volatile("mbarrier.arrive.release.cta.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_st_32x32b_x32_l(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]),
      "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]),
      "r"(r[30]), "r"(r[31])
      : "memory");
}
// tab[h, clamp(delta, -R, R)]: the table is constant beyond the radius, so this equals tab[h, delta] wherever delta is valid,
// and stays inside the table for the out-of-range deltas of padded rows / keys past T (whose results are never used)
__device__ __forceinline__ float tab_at(const float* tab_h, int T, int R, int delta) {
  return __ldg(tab_h + (min(max(delta, -R), R) + T - 1));
}

constexpr int kLongMaxT = 16384;

// ------------------------------------------------------------------------------------------------ forward
constexpr int kLfQ = 0, kLfK = 32768, kLfV = 65536, kLfP = 98304, kLfRing = 163840;   // Q / K / V / P as in attn_fwd.cu
constexpr int kLfThreads = 320;
constexpr int kLfCopies = 4;
constexpr int kLfWin = 384;                     // table entries one key tile needs for 256 query rows: 128 + 256 - 1, rounded up
constexpr int kLfCopyStride = kLfWin + 8;       // copies start 8 banks apart (conflict-free 128-bit loads, see attn_fwd.cu)
constexpr int kLfStage = kLfCopies * kLfCopyStride + kAttnTile;  // floats per ring stage: 4 table copies + the key mask
constexpr int kLfSmem = kLfRing + 2 * kLfStage * 4 + 1024;       // the same for every T
constexpr float kLfRebase = 1.2089258e24f;      // 2^80, as in attn_fwd.cu

__global__ void __launch_bounds__(kLfThreads, 1) attn_fwd_long_kernel(const __grid_constant__ CUtensorMap tm,
                                                                      const __grid_constant__ AttnParams p, int R) {
  pdl_grid_sync();
  const int tid = threadIdx.x, warp = tid >> 5;
  const int wg = warp >> 2;
  const int q0 = blockIdx.x * 2 * kAttnTile, h = blockIdx.y, b = blockIdx.z;
  const int T = p.T, D = p.D, N = p.n_tiles;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* sQ = smem + kLfQ;
  uint8_t* sK = smem + kLfK;
  uint8_t* sV = smem + kLfV;
  uint8_t* sP = smem + kLfP;
  float* ring = reinterpret_cast<float*>(smem + kLfRing);  // [2][kLfStage]

  __shared__ uint64_t q_full, k_full[2], k_empty[2], v_full[2], v_empty[2], s_full[2], p_ready[2], pv_done[2], w_full[2],
      w_empty[2];
  __shared__ uint32_t tmem_base_s;
  __shared__ int n_eff_s, wmask_s[2];

  // ---- key padding: number of key tiles holding a valid key, and whether any of the CTA's 256 query rows is live.  One
  // pass over the utterance's pad bytes, no per-key storage.
  int n_eff = N;
  if (p.key_pad != nullptr) {
    if (tid == 0) n_eff_s = 1;
    __syncthreads();
    const uint8_t* kp = p.key_pad + static_cast<long long>(b) * T;
    int last_valid = -1, live = 0;
    for (int j = tid; j < T; j += kLfThreads) {
      if (kp[j] == 0) {
        last_valid = j;
        if (j >= q0 && j < q0 + 2 * kAttnTile) live = 1;
      }
    }
    if (last_valid >= 0) atomicMax(&n_eff_s, last_valid / kAttnTile + 1);
    if (!__syncthreads_or(live)) {  // all 256 query rows padded: zeros, as attn_fwd.cu
      if (tid < 2 * kAttnTile && q0 + tid < T) {
        uint4* dst = reinterpret_cast<uint4*>(p.out + (static_cast<long long>(b) * T + q0 + tid) * D + h * kHeadDim);
#pragma unroll
        for (int g = 0; g < 8; ++g) dst[g] = make_uint4(0u, 0u, 0u, 0u);
        if (p.lse != nullptr) p.lse[(static_cast<long long>(b) * p.H + h) * T + q0 + tid] = INFINITY;
      }
      return;
    }
    n_eff = n_eff_s;
  }

  if (warp == 8 && (tid & 31) == 0) {
    tma_prefetch_desc(&tm);
    mbar_init(&q_full, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&k_full[i], 1);
      mbar_init(&v_full[i], 1);
      mbar_init(&k_empty[i], 1);
      mbar_init(&v_empty[i], 1);
      mbar_init(&s_full[i], 1);
      mbar_init(&pv_done[i], 1);
      mbar_init(&p_ready[i], kAttnTile);
      mbar_init(&w_full[i], 32);   // every lane of the TMA warp, after writing its share of the window
      mbar_init(&w_empty[i], 8);   // one lane per softmax warp, after its last read of the window
    }
    fence_mbar_init();
    mbar_expect_tx(&q_full, 32768);
    tma_load_4d(sQ, &tm, &q_full, h * kHeadDim, q0, b, 0);
    tma_load_4d(sQ + 16384, &tm, &q_full, h * kHeadDim, q0 + kAttnTile, b, 0);
    mbar_expect_tx(&k_full[0], 16384);
    tma_load_4d(sK, &tm, &k_full[0], D + h * kHeadDim, 0, b, 0);
    mbar_expect_tx(&v_full[0], 16384);
    tma_load_4d(sV, &tm, &v_full[0], 2 * D + h * kHeadDim, 0, b, 0);
  }
  __syncwarp();
  if (warp == 0) tmem_alloc(&tmem_base_s, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;
  const float* tab_h = p.tab + static_cast<long long>(h) * (2 * T - 1);

  if (warp == 8) {
    // ------------------------------------------------------------------ TMA warp: K / V tiles (lane 0) and, with all 32
    // lanes, the table window and key mask of every key tile
    const int lane = tid & 31;
    const uint8_t* kp = p.key_pad != nullptr ? p.key_pad + static_cast<long long>(b) * T : nullptr;
    for (int n = 0; n < n_eff; ++n) {
      const int s = n & 1;
      const uint32_t ph = (n >> 1) & 1;
      const int k0 = n * kAttnTile;
      if (lane == 0 && n >= 1) {
        mbar_wait(&k_empty[s], ph ^ 1);
        mbar_expect_tx(&k_full[s], 16384);
        tma_load_4d(sK + s * 16384, &tm, &k_full[s], D + h * kHeadDim, k0, b, 0);
      }
      mbar_wait(&w_empty[s], ph ^ 1);
      float* w = ring + s * kLfStage;
      // window entry m <-> delta = dlo + m; copy c holds entry k + c at index k
      const int dlo = k0 - q0 - (2 * kAttnTile - 1);
      const bool cta_far = dlo >= R || k0 + kAttnTile - 1 - q0 <= -R;
      if (!cta_far) {
        for (int m = lane; m < kLfWin + kLfCopies - 1; m += 32) {
          const float v = tab_at(tab_h, T, R, dlo + m);
#pragma unroll
          for (int c = 0; c < kLfCopies; ++c)
            if (m - c >= 0 && m - c < kLfWin) w[c * kLfCopyStride + m - c] = v;
        }
      }
      bool any = false;
#pragma unroll
      for (int c = lane; c < kAttnTile; c += 32) {
        const int j = k0 + c;
        const bool masked = j >= T || (kp != nullptr && kp[j] != 0);
        w[kLfCopies * kLfCopyStride + c] = masked ? -INFINITY : 0.f;
        any |= masked;
      }
      any = __any_sync(0xffffffffu, any);
      if (lane == 0) wmask_s[s] = any ? 1 : 0;
      mbar_arrive_rel_l(&w_full[s]);
      if (lane == 0 && n >= 1) {
        mbar_wait(&v_empty[s], ph ^ 1);
        mbar_expect_tx(&v_full[s], 16384);
        tma_load_4d(sV + s * 16384, &tm, &v_full[s], 2 * D + h * kHeadDim, k0, b, 0);
      }
      __syncwarp();
    }
  } else if (warp == 9) {
    // ------------------------------------------------------------------ MMA-issuing warp, as attn_fwd.cu
    if ((tid & 31) == 0) {
      constexpr uint32_t idesc_s = make_idesc_bf16(128, 128, 0, 0);
      constexpr uint32_t idesc_pv = make_idesc_bf16(128, 64, 0, 1);
      auto issue_s = [&](int w, int n) {
        const uint32_t a = smem_u32(sQ + w * 16384), bb = smem_u32(sK + (n & 1) * 16384);
#pragma unroll
        for (int k = 0; k < 4; ++k)
          umma_bf16(tmem + w * 256, make_smem_desc_sw128(a + k * 32, 16, 1024), make_smem_desc_sw128(bb + k * 32, 16, 1024),
                    idesc_s, k > 0 ? 1u : 0u);
        umma_commit(&s_full[w]);
      };
      mbar_wait(&q_full, 0);
      mbar_wait(&k_full[0], 0);
      tc_fence_after();
      issue_s(0, 0);
      issue_s(1, 0);
      umma_commit(&k_empty[0]);
      for (int n = 0; n < n_eff; ++n) {
#pragma unroll 1
        for (int w = 0; w < 2; ++w) {
          mbar_wait(&p_ready[w], n & 1);
          tc_fence_after();
          if (n + 1 < n_eff) {
            if (w == 0) {
              mbar_wait(&k_full[(n + 1) & 1], ((n + 1) >> 1) & 1);
              tc_fence_after();
            }
            issue_s(w, n + 1);
            if (w == 1) umma_commit(&k_empty[(n + 1) & 1]);
          }
          if (w == 0) {
            mbar_wait(&v_full[n & 1], (n >> 1) & 1);
            tc_fence_after();
          }
          const uint32_t a = smem_u32(sP + w * 32768), bb = smem_u32(sV + (n & 1) * 16384);
#pragma unroll
          for (int k = 0; k < 8; ++k)
            umma_bf16(tmem + w * 256 + 128, make_smem_desc_sw128(a + (k >> 2) * 16384 + (k & 3) * 32, 16, 1024),
                      make_smem_desc_sw128(bb + k * 2048, 8192, 1024), idesc_pv, (n > 0 || k > 0) ? 1u : 0u);
          umma_commit(&pv_done[w]);
          if (w == 1) umma_commit(&v_empty[n & 1]);
        }
      }
    }
  } else {
    // ------------------------------------------------------------------ softmax warpgroups
    const int r = tid & 127;
    const int r256 = wg * kAttnTile + r;
    const int lane = tid & 31;
    const bool row_valid = (q0 + r256) < T;
    const uint32_t lane_addr = static_cast<uint32_t>((warp & 3) * 32) << 16;
    const uint32_t s_addr = tmem + wg * 256 + lane_addr;
    const uint32_t o_addr = tmem + wg * 256 + 128 + lane_addr;
    uint8_t* sPw = sP + wg * 32768;

    const float g = (p.gate != nullptr && row_valid) ? p.gate[(static_cast<long long>(b) * p.H + h) * T + q0 + r256] : 1.0f;
    const float gl = g * kLog2e;
    const float sc = p.scale * kLog2e;
    const int toff = 2 * kAttnTile - 1 - r256;  // this row's first window entry (key k0): m = c + 255 - r256
    const int wrow0 = q0 + wg * kAttnTile;      // first query row of this warpgroup

    float m_ref = -INFINITY, l_run = 0.f;

    for (int n = 0; n < n_eff; ++n) {
      const int s = n & 1;
      const int k0 = n * kAttnTile;
      mbar_wait(&s_full[wg], n & 1);
      tc_fence_after();
      mbar_wait(&w_full[s], (n >> 1) & 1);
      const float* w = ring + s * kLfStage;
      const float4* tab4 = reinterpret_cast<const float4*>(w + (toff & 3) * kLfCopyStride + (toff & ~3));
      const float* kbias = w + kLfCopies * kLfCopyStride;
      const bool msk = wmask_s[s] != 0;
      // off band for this warpgroup's 128 rows: one per-row constant replaces the table
      const bool far_p = k0 - (wrow0 + kAttnTile - 1) >= R, far_n = k0 + kAttnTile - 1 - wrow0 <= -R;
      const bool band = !(far_p || far_n);
      const float cbias = band ? 0.f : gl * __ldg(tab_h + (T - 1 + (far_p ? R : -R)));

      auto tile_max = [&]() {
        float mx = -INFINITY;
#pragma unroll 1
        for (int c0 = 0; c0 < kAttnTile; c0 += 32) {
          uint32_t su[32];
          tmem_ld_32x32b_x32(s_addr + c0, su);
          tmem_ld_wait();
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            const float4 tb = band ? tab4[c0 / 4 + q] : make_float4(0.f, 0.f, 0.f, 0.f);
            float x0 = fmaf(__uint_as_float(su[4 * q]), sc, cbias), x1 = fmaf(__uint_as_float(su[4 * q + 1]), sc, cbias);
            float x2 = fmaf(__uint_as_float(su[4 * q + 2]), sc, cbias), x3 = fmaf(__uint_as_float(su[4 * q + 3]), sc, cbias);
            x0 = fmaf(gl, tb.x, x0); x1 = fmaf(gl, tb.y, x1); x2 = fmaf(gl, tb.z, x2); x3 = fmaf(gl, tb.w, x3);
            if (msk) {
              const float4 kb = *reinterpret_cast<const float4*>(kbias + c0 + 4 * q);
              x0 += kb.x; x1 += kb.y; x2 += kb.z; x3 += kb.w;
            }
            mx = fmaxf(fmaxf(mx, fmaxf(x0, x1)), fmaxf(x2, x3));
          }
        }
        return mx;
      };

      if (__any_sync(0xffffffffu, m_ref == -INFINITY)) {
        const float mx = tile_max();
        if (m_ref == -INFINITY) m_ref = mx;
      }
      bool p_free = (n == 0);
      auto softmax_tile = [&](auto MSK, auto BAND) -> float {
        constexpr bool kMsk = decltype(MSK)::value;
        constexpr bool kBand = decltype(BAND)::value;
        const float neg_ref = ((m_ref == -INFINITY) ? 0.f : -m_ref) + (kBand ? 0.f : cbias);
        float part0 = 0.f, part1 = 0.f, part2 = 0.f, part3 = 0.f;
        uint32_t sa[32], sb[32];
        tmem_ld_32x32b_x32(s_addr, sa);
        tmem_ld_wait();
#pragma unroll
        for (int cc = 0; cc < 4; ++cc) {
          const int c0 = cc * 32;
          uint32_t* su = (cc & 1) ? sb : sa;
          if (cc + 1 < 4) tmem_ld_32x32b_x32(s_addr + c0 + 32, (cc & 1) ? sa : sb);
          float pv[32];
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            float4 tb = make_float4(0.f, 0.f, 0.f, 0.f), kb = make_float4(0.f, 0.f, 0.f, 0.f);
            if (kBand) tb = tab4[c0 / 4 + q];
            if (kMsk) kb = *reinterpret_cast<const float4*>(kbias + c0 + 4 * q);
            const float tbv[4] = {tb.x, tb.y, tb.z, tb.w};
            const float kbv[4] = {kb.x, kb.y, kb.z, kb.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const int j = 4 * q + e;
              float x = fmaf(__uint_as_float(su[j]), sc, neg_ref);
              if (kBand) x = fmaf(gl, tbv[e], x);
              if (kMsk) x += kbv[e];
              const float ex = fast_exp2_l(x);
              if (e == 0) part0 += ex; else if (e == 1) part1 += ex; else if (e == 2) part2 += ex; else part3 += ex;
              pv[j] = ex;
            }
          }
          if (!p_free) {
            mbar_wait(&pv_done[wg], (n - 1) & 1);
            p_free = true;
          }
#pragma unroll
          for (int gq = 0; gq < 4; ++gq) {
            uint4 wv;
            wv.x = pack_bf16x2(pv[gq * 8 + 0], pv[gq * 8 + 1]);
            wv.y = pack_bf16x2(pv[gq * 8 + 2], pv[gq * 8 + 3]);
            wv.z = pack_bf16x2(pv[gq * 8 + 4], pv[gq * 8 + 5]);
            wv.w = pack_bf16x2(pv[gq * 8 + 6], pv[gq * 8 + 7]);
            store_sw128_chunk(sPw, r, (c0 >> 3) + gq, wv);
          }
          if (cc + 1 < 4) tmem_ld_wait();
        }
        return (part0 + part1) + (part2 + part3);
      };
      float lsum;
#pragma unroll 1
      while (true) {
        if (band) lsum = msk ? softmax_tile(std::true_type{}, std::true_type{}) : softmax_tile(std::false_type{}, std::true_type{});
        else lsum = msk ? softmax_tile(std::true_type{}, std::false_type{}) : softmax_tile(std::false_type{}, std::false_type{});
        if (!__any_sync(0xffffffffu, !(lsum < kLfRebase))) break;
        // re-base (rare), as attn_fwd.cu
        const float m_new = fmaxf(m_ref, tile_max());
        const float factor = (m_ref == -INFINITY) ? 0.f : fast_exp2_l(m_ref - m_new);
        if (n >= 1) {
          mbar_wait(&pv_done[wg], (n - 1) & 1);
          p_free = true;
          tc_fence_after();
          uint32_t t0[32];
#pragma unroll 1
          for (int hlf = 0; hlf < 2; ++hlf) {
            tmem_ld_32x32b_x32(o_addr + hlf * 32, t0);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 32; ++i) t0[i] = __float_as_uint(__uint_as_float(t0[i]) * factor);
            tmem_st_32x32b_x32_l(o_addr + hlf * 32, t0);
          }
          asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        }
        l_run *= factor;
        m_ref = m_new;
      }
      l_run += lsum;
      __syncwarp();
      if (lane == 0) mbar_arrive(&w_empty[s]);  // this warp is done with the window and mask of tile n

      fence_proxy_async_smem();
      tc_fence_before();
      mbar_arrive_rel_l(&p_ready[wg]);
    }
    mbar_wait(&pv_done[wg], (n_eff - 1) & 1);
    tc_fence_after();

    uint32_t t0[32], t1[32];
    tmem_ld_32x32b_x32(o_addr, t0);
    tmem_ld_32x32b_x32(o_addr + 32, t1);
    tmem_ld_wait();
    if (row_valid) {
      const float inv = l_run > 0.f ? 1.0f / l_run : 0.f;
      __nv_bfloat16* dst = p.out + (static_cast<long long>(b) * T + q0 + r256) * D + h * kHeadDim;
#pragma unroll
      for (int gq = 0; gq < 4; ++gq) {
        uint4 wv;
        wv.x = pack_bf16x2(__uint_as_float(t0[gq * 8 + 0]) * inv, __uint_as_float(t0[gq * 8 + 1]) * inv);
        wv.y = pack_bf16x2(__uint_as_float(t0[gq * 8 + 2]) * inv, __uint_as_float(t0[gq * 8 + 3]) * inv);
        wv.z = pack_bf16x2(__uint_as_float(t0[gq * 8 + 4]) * inv, __uint_as_float(t0[gq * 8 + 5]) * inv);
        wv.w = pack_bf16x2(__uint_as_float(t0[gq * 8 + 6]) * inv, __uint_as_float(t0[gq * 8 + 7]) * inv);
        *reinterpret_cast<uint4*>(dst + gq * 8) = wv;
      }
#pragma unroll
      for (int gq = 0; gq < 4; ++gq) {
        uint4 wv;
        wv.x = pack_bf16x2(__uint_as_float(t1[gq * 8 + 0]) * inv, __uint_as_float(t1[gq * 8 + 1]) * inv);
        wv.y = pack_bf16x2(__uint_as_float(t1[gq * 8 + 2]) * inv, __uint_as_float(t1[gq * 8 + 3]) * inv);
        wv.z = pack_bf16x2(__uint_as_float(t1[gq * 8 + 4]) * inv, __uint_as_float(t1[gq * 8 + 5]) * inv);
        wv.w = pack_bf16x2(__uint_as_float(t1[gq * 8 + 6]) * inv, __uint_as_float(t1[gq * 8 + 7]) * inv);
        *reinterpret_cast<uint4*>(dst + 32 + gq * 8) = wv;
      }
      if (p.lse != nullptr)
        p.lse[(static_cast<long long>(b) * p.H + h) * T + q0 + r256] = (l_run > 0.f) ? (m_ref + log2f(l_run)) : INFINITY;
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    __syncwarp();
    tmem_dealloc(tmem, 512);
  }
}

// ------------------------------------------------------------------------------------------------ backward: dK / dV
// As attn_bwd.cu's dK/dV kernel (CTA = 128 keys, thread = key row, loop over query tiles); the table window of query tile qi
// is staged with that tile's column vector: win[l] = tab[h, k0 - i0 - 127 + l], element (key r, query column c) at l = r - c + 127.
constexpr int kLkK = 0, kLkV = 16384, kLkQ = 32768, kLkDO = 65536, kLkPT = 98304, kLkDST = 131072, kLkVec = 163840,
              kLkWin = 167936;
constexpr int kLkSmem = kLkWin + 2 * 256 * 4 + 1024;

template <bool HAS_BIAS>
__global__ void __launch_bounds__(256, 1) attn_bwd_dkv_long_kernel(const __grid_constant__ CUtensorMap tm_qkv,
                                                                   const __grid_constant__ CUtensorMap tm_do,
                                                                   const __grid_constant__ AttnParams p, int R) {
  pdl_grid_sync();
  const int tid = threadIdx.x, warp = tid >> 5;
  const int k0 = blockIdx.x * kAttnTile, h = blockIdx.y, b = blockIdx.z;
  const int T = p.T, D = p.D, N = p.n_tiles;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* sK = smem + kLkK;
  uint8_t* sV = smem + kLkV;
  uint8_t* sQ = smem + kLkQ;
  uint8_t* sDO = smem + kLkDO;
  uint8_t* sPT = smem + kLkPT;
  uint8_t* sDST = smem + kLkDST;
  float4* colvec = reinterpret_cast<float4*>(smem + kLkVec);  // [2][128] {lse2, delta, gate*log2e, unused}
  float* win = reinterpret_cast<float*>(smem + kLkWin);       // [2][256]

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

  const float* tab_h = HAS_BIAS ? p.tab + static_cast<long long>(h) * (2 * T - 1) : nullptr;
  auto load_tile_vecs = [&](int qi) {  // column vector and table window of query tile qi
    const int i0 = qi * kAttnTile;
    if (HAS_BIAS && tid < 2 * kAttnTile - 1) {
      const int dlo = k0 - i0 - (kAttnTile - 1);
      const bool far = dlo >= R || dlo + 2 * kAttnTile - 2 <= -R;
      // off band every entry is tab[+-R]: one broadcast address instead of 255
      win[(qi & 1) * 256 + tid] = tab_at(tab_h, T, R, far ? dlo : dlo + tid);
    }
    if (tid >= kAttnTile) return;
    const int i = i0 + tid;
    float4 v;
    if (i < T) {
      const long long idx = (static_cast<long long>(b) * p.H + h) * T + i;
      v.x = p.lse[idx];
      v.y = p.delta[idx];
      v.z = (HAS_BIAS ? ((p.gate != nullptr) ? p.gate[idx] : 1.0f) : 0.f) * kLog2e;
    } else {
      v.x = INFINITY;
      v.y = 0.f;
      v.z = 0.f;
    }
    v.w = 0.f;
    colvec[(qi & 1) * kAttnTile + tid] = v;
  };
  load_tile_vecs(0);
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
  auto issue_st = [&](int qi) {
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

  const int r = tid & (kAttnTile - 1);
  const int half = tid >> 7;
  const int key = k0 + r;
  const bool key_valid = key < T;
  const bool key_masked = !key_valid || (p.key_pad != nullptr && p.key_pad[static_cast<long long>(b) * T + key] != 0);
  const float kb = key_masked ? -INFINITY : 0.f;
  const float sc = p.scale * kLog2e;
  const uint32_t lane_addr = static_cast<uint32_t>((warp & 3) * 32) << 16;

  for (int qi = 0; qi < N; ++qi) {
    const int st = qi & 1;
    mbar_wait(&st_full, qi & 1);
    tc_fence_after();
    if (tid == 0 && qi >= 1 && qi + 1 < N) load_qdo(qi + 1);
    __syncwarp();
    const float4* cv = colvec + st * kAttnTile;
    const float* tabrow = win + st * 256 + r + kAttnTile - 1;
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
        if (HAS_BIAS) x = fmaf(c.z, tabrow[-(c0 + j)], x);
        const float pr = fast_exp2_l(x - c.x);
        pv[j] = pr;
        dv[j] = pr * (__uint_as_float(du[j]) - c.y) * p.scale;
      }
#pragma unroll
      for (int gq = 0; gq < 4; ++gq) {
        uint4 w;
        w.x = pack_bf16x2(pv[gq * 8 + 0], pv[gq * 8 + 1]);
        w.y = pack_bf16x2(pv[gq * 8 + 2], pv[gq * 8 + 3]);
        w.z = pack_bf16x2(pv[gq * 8 + 4], pv[gq * 8 + 5]);
        w.w = pack_bf16x2(pv[gq * 8 + 6], pv[gq * 8 + 7]);
        store_sw128_chunk(sPT, r, (c0 >> 3) + gq, w);
        w.x = pack_bf16x2(dv[gq * 8 + 0], dv[gq * 8 + 1]);
        w.y = pack_bf16x2(dv[gq * 8 + 2], dv[gq * 8 + 3]);
        w.z = pack_bf16x2(dv[gq * 8 + 4], dv[gq * 8 + 5]);
        w.w = pack_bf16x2(dv[gq * 8 + 6], dv[gq * 8 + 7]);
        store_sw128_chunk(sDST, r, (c0 >> 3) + gq, w);
      }
    }
    if (qi + 1 < N) load_tile_vecs(qi + 1);
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    if (tid == 0) {
      tc_fence_after();
      const uint32_t apt = smem_u32(sPT), ads = smem_u32(sDST), bdo = smem_u32(sDO + st * 16384),
                     bq = smem_u32(sQ + st * 16384);
#pragma unroll
      for (int k = 0; k < 8; ++k) {
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
    const uint32_t col = 256 + half * 64;  // warpgroup 0 writes dV, warpgroup 1 dK
    tmem_ld_32x32b_x32(tmem + lane_addr + col, t0);
    tmem_ld_32x32b_x32(tmem + lane_addr + col + 32, t1);
    tmem_ld_wait();
    if (key_valid) {
      __nv_bfloat16* dst = p.dqkv + (static_cast<long long>(b) * T + key) * (3 * D) + (half == 0 ? 2 * D : D) + h * kHeadDim;
#pragma unroll
      for (int gq = 0; gq < 4; ++gq) {
        uint4 w;
        w.x = pack_bf16x2(__uint_as_float(t0[gq * 8 + 0]), __uint_as_float(t0[gq * 8 + 1]));
        w.y = pack_bf16x2(__uint_as_float(t0[gq * 8 + 2]), __uint_as_float(t0[gq * 8 + 3]));
        w.z = pack_bf16x2(__uint_as_float(t0[gq * 8 + 4]), __uint_as_float(t0[gq * 8 + 5]));
        w.w = pack_bf16x2(__uint_as_float(t0[gq * 8 + 6]), __uint_as_float(t0[gq * 8 + 7]));
        *reinterpret_cast<uint4*>(dst + gq * 8) = w;
        w.x = pack_bf16x2(__uint_as_float(t1[gq * 8 + 0]), __uint_as_float(t1[gq * 8 + 1]));
        w.y = pack_bf16x2(__uint_as_float(t1[gq * 8 + 2]), __uint_as_float(t1[gq * 8 + 3]));
        w.z = pack_bf16x2(__uint_as_float(t1[gq * 8 + 4]), __uint_as_float(t1[gq * 8 + 5]));
        w.w = pack_bf16x2(__uint_as_float(t1[gq * 8 + 6]), __uint_as_float(t1[gq * 8 + 7]));
        *reinterpret_cast<uint4*>(dst + 32 + gq * 8) = w;
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

// ------------------------------------------------------------------------------------------------ backward: dQ / d gate / d tab
// As attn_bwd.cu's dQ kernel (CTA = 128 queries, thread = query row, loop over key tiles).  Per key tile n, the table window
// win[l] = tab[h, k0 - q0 - 127 + l] (element (row r, key column c) at l = c - r + 127) and the tile's key mask are staged
// double-buffered; whether the tile has a masked key comes out of the barrier that separates two tiles (__syncthreads_or).
// d tab of a band tile: diagonal sums of the staged gate * dS tile into a 255-entry window, flushed with atomics at the end of
// the tile.  Off-band tiles: each row sums its dS over the tile; gate_i times that sum goes to d tab at delta = +-R.
constexpr int kLqQ = 0, kLqDO = 16384, kLqK = 32768, kLqV = 65536, kLqDS = 98304, kLqW = 131072;
constexpr int kLqWStride = 130;  // as attn_bwd.cu
constexpr int kLqWin = kLqW + 128 * kLqWStride * 2 + 64;  // [2][256] table windows, [2][128] key masks, [256] d tab window
constexpr int kLqSmem = kLqWin + (2 * 256 + 2 * 128 + 256) * 4 + 1024;

template <bool HAS_BIAS>
__global__ void __launch_bounds__(256, 1) attn_bwd_dq_long_kernel(const __grid_constant__ CUtensorMap tm_qkv,
                                                                  const __grid_constant__ CUtensorMap tm_do,
                                                                  const __grid_constant__ AttnParams p, int R) {
  pdl_grid_sync();
  const int tid = threadIdx.x, warp = tid >> 5;
  const int q0 = blockIdx.x * kAttnTile, h = blockIdx.y, b = blockIdx.z;
  const int T = p.T, D = p.D, N = p.n_tiles;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* sQ = smem + kLqQ;
  uint8_t* sDO = smem + kLqDO;
  uint8_t* sK = smem + kLqK;
  uint8_t* sV = smem + kLqV;
  uint8_t* sDS = smem + kLqDS;
  __nv_bfloat16* sW = reinterpret_cast<__nv_bfloat16*>(smem + kLqW);
  float* win = reinterpret_cast<float*>(smem + kLqWin);  // [2][256]
  float* kmask = win + 2 * 256;                          // [2][128]
  float* dwin = kmask + 2 * kAttnTile;                   // [256]

  __shared__ uint64_t qdo_full, kv_full[2], s_full, acc_done;
  __shared__ uint32_t tmem_base_s;
  __shared__ float far_acc[2];

  if (tid == 0) {
    tma_prefetch_desc(&tm_qkv);
    tma_prefetch_desc(&tm_do);
    mbar_init(&qdo_full, 1);
    mbar_init(&kv_full[0], 1);
    mbar_init(&kv_full[1], 1);
    mbar_init(&s_full, 1);
    mbar_init(&acc_done, 1);
    fence_mbar_init();
    far_acc[0] = far_acc[1] = 0.f;
  }
  __syncwarp();
  if (warp == 0) tmem_alloc(&tmem_base_s, 512);

  const float* tab_h = HAS_BIAS ? p.tab + static_cast<long long>(h) * (2 * T - 1) : nullptr;
  const uint8_t* kp = p.key_pad != nullptr ? p.key_pad + static_cast<long long>(b) * T : nullptr;
  auto tile_far = [&](int n, int& sign) {  // +1 / -1: every pair of tile n has delta >= R / <= -R; 0: band
    const int dlo = n * kAttnTile - q0 - (kAttnTile - 1);
    sign = dlo >= R ? 1 : (dlo + 2 * kAttnTile - 2 <= -R ? -1 : 0);
    return sign != 0;
  };
  // stages tile n's table window (band tiles) and key mask; returns this thread's "masked key" bit
  auto load_tile_vecs = [&](int n) -> int {
    const int k0 = n * kAttnTile;
    int sign;
    if (HAS_BIAS && !tile_far(n, sign) && tid < 2 * kAttnTile - 1)
      win[(n & 1) * 256 + tid] = tab_at(tab_h, T, R, k0 - q0 - (kAttnTile - 1) + tid);
    if (tid >= kAttnTile) return 0;
    const int j = k0 + tid;
    const bool masked = j >= T || (kp != nullptr && kp[j] != 0);
    kmask[(n & 1) * kAttnTile + tid] = masked ? -INFINITY : 0.f;
    return masked ? 1 : 0;
  };
  int msk_next = load_tile_vecs(0);
  if (HAS_BIAS) dwin[tid] = 0.f;
  tc_fence_before();
  msk_next = __syncthreads_or(msk_next);
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
  auto issue_s = [&](int n) {
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

  const int r = tid & (kAttnTile - 1);
  const int half = tid >> 7;
  const bool row_valid = (q0 + r) < T;
  const long long ridx = (static_cast<long long>(b) * p.H + h) * T + q0 + r;
  const float lse2 = row_valid ? p.lse[ridx] : INFINITY;
  const float delta = row_valid ? p.delta[ridx] : 0.f;
  float g = 0.f;
  if (HAS_BIAS) g = (p.gate != nullptr && row_valid) ? p.gate[ridx] : (row_valid ? 1.0f : 0.f);
  const float gl = g * kLog2e;
  const float sc = p.scale * kLog2e;
  const float t_pos = HAS_BIAS ? __ldg(tab_h + R + T - 1) : 0.f, t_neg = HAS_BIAS ? __ldg(tab_h + (T - 1 - R)) : 0.f;
  const uint32_t lane_addr = static_cast<uint32_t>((warp & 3) * 32) << 16;
  float dgate_acc = 0.f, far_pos = 0.f, far_neg = 0.f;  // far_*: sum of this row's dS over off-band tiles
  uint32_t* wrow = reinterpret_cast<uint32_t*>(sW) + r * (kLqWStride / 2);

  for (int n = 0; n < N; ++n) {
    const int st = n & 1;
    const int k0 = n * kAttnTile;
    mbar_wait(&s_full, n & 1);
    tc_fence_after();
    if (tid == 0 && n >= 1 && n + 1 < N) load_kv(n + 1);
    __syncwarp();
    const bool msk = msk_next != 0;
    int sign = 0;
    const bool far = HAS_BIAS && tile_far(n, sign);
    const float* tabrow = win + st * 256 + (kAttnTile - 1 - r);
    const float* kb = kmask + st * kAttnTile;
    const float tfar = sign > 0 ? t_pos : t_neg;
    float ds_sum = 0.f;
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
          tb = far ? tfar : tabrow[c0 + j];
          x = fmaf(gl, tb, x);
        }
        if (msk) x += kb[c0 + j];
        const float pr = fast_exp2_l(x - lse2);
        const float ds = pr * (__uint_as_float(du[j]) - delta);
        if (HAS_BIAS) dgate_acc = fmaf(ds, tb, dgate_acc);
        ds_sum += ds;
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
      if (HAS_BIAS && !far) {
#pragma unroll
        for (int j = 0; j < 16; ++j) wrow[(c0 >> 1) + j] = pack_bf16x2(g * dsv[2 * j], g * dsv[2 * j + 1]);
      }
    }
    if (HAS_BIAS && far) {
      if (sign > 0) far_pos += ds_sum; else far_neg += ds_sum;
    }
    const int msk_bit = (n + 1 < N) ? load_tile_vecs(n + 1) : 0;
    fence_proxy_async_smem();
    tc_fence_before();
    msk_next = __syncthreads_or(msk_bit);
    if (tid == 0) {
      tc_fence_after();
      const uint32_t ads = smem_u32(sDS), bk = smem_u32(sK + st * 16384);
#pragma unroll
      for (int k = 0; k < 8; ++k) {
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
    if (HAS_BIAS && !far) {
      // diagonal sums of the staged tile (as attn_bwd.cu): thread d sums W[rr][(rr+d) & 127] over its half's rows;
      // diagonal c - rr = d is window entry d + 127, the wrapped one (c - rr = d - 128) entry d - 1
      const int d = r;
      float acc_pos = 0.f, acc_neg = 0.f;
#pragma unroll 8
      for (int rr = half * 64; rr < half * 64 + 64; ++rr) {
        const int c = (rr + d) & (kAttnTile - 1);
        const float v = __bfloat162float(sW[rr * kLqWStride + c]);
        if (rr + d < kAttnTile) acc_pos += v; else acc_neg += v;
      }
      atomicAdd(&dwin[d + kAttnTile - 1], acc_pos);
      if (d > 0) atomicAdd(&dwin[d - 1], acc_neg);
      __syncthreads();  // sW is rewritten by the next tile; dwin is complete
      if (p.dtab != nullptr && tid < 2 * kAttnTile - 1) {
        const float v = dwin[tid];
        const int dl = min(max(k0 - q0 - (kAttnTile - 1) + tid, -R), R);
        if (v != 0.f) atomicAdd(p.dtab + static_cast<long long>(h) * (2 * T - 1) + dl + T - 1, v);
      }
      dwin[tid] = 0.f;  // (re-written after the next tile's first barrier)
    }
  }
  mbar_wait(&acc_done, 0);
  tc_fence_after();
  {
    uint32_t t0[32];
    tmem_ld_32x32b_x32(tmem + lane_addr + 256 + half * 32, t0);
    tmem_ld_wait();
    __shared__ float dgate_x[kAttnTile];
    if (HAS_BIAS) {
      // off-band d tab: sum over the CTA's rows of gate_i * (row's off-band dS sum), one atomic per side
      const float fp = warp_sum(g * far_pos), fn = warp_sum(g * far_neg);
      if ((tid & 31) == 0) {
        if (fp != 0.f) atomicAdd(&far_acc[0], fp);
        if (fn != 0.f) atomicAdd(&far_acc[1], fn);
      }
      if (half == 1) dgate_x[r] = dgate_acc;
    }
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
    if (HAS_BIAS && p.dtab != nullptr && tid < 2) {
      const float v = far_acc[tid];
      if (v != 0.f) atomicAdd(p.dtab + static_cast<long long>(h) * (2 * T - 1) + (tid == 0 ? T - 1 + R : T - 1 - R), v);
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
cudaError_t launch_attn_delta(const void* out, const void* dout, int B, int T, int H, float* delta, cudaStream_t st);

// shapes both long kernels accept: every index the kernels form past a 32-bit int is taken in 64 bits; what stays 32-bit is
// the grid (H, B <= 65535), the TMA coordinates (< T) and the table index (< 2T - 1)
static int check_long_shape(const char* who, int B, int T, int H, int R, bool has_bias) {
  B200_CHECK_ARG(T >= 1 && T <= kLongMaxT, "%s: T=%d out of range (1..%d)", who, T, kLongMaxT);
  B200_CHECK_ARG(B >= 1 && B <= 65535 && H >= 1 && H <= 65535, "%s: B=%d, H=%d out of range (1..65535)", who, B, H);
  B200_CHECK_ARG(!has_bias || (R >= 0 && R <= T - 1), "%s: tab_radius=%d out of range (0..T-1=%d)", who, R, T - 1);
  // the bf16 [B,T,3D] operand is addressed by TMA with 64-bit strides, and its row count B*T by the delta pre-kernel's grid
  B200_CHECK_ARG(static_cast<long long>(B) * T * 32 / 256 < (1LL << 31), "%s: B*T=%lld too large", who,
                 static_cast<long long>(B) * T);
  return 0;
}

}  // namespace b200

using namespace b200;

extern "C" {

int b200s_attn_fwd_long(const void* qkv, const float* gate, const float* tab, int tab_radius, const uint8_t* key_pad, void* out,
                        float* lse, int B, int T, int H, float scale, b200s_stream stream) {
  B200_CHECK_ARG(qkv && tab && out, "attn_fwd_long: null pointer (the table is required)");
  if (int rc = check_long_shape("attn_fwd_long", B, T, H, tab_radius, true)) return rc;
  const int D = H * kHeadDim;
  CUtensorMap tm;
  if (make_qkv_tmap(&tm, qkv, T, B, 3 * D, kAttnTile)) return -3;
  AttnParams p;
  memset(&p, 0, sizeof(p));
  p.T = T; p.H = H; p.B = B; p.D = D;
  p.n_tiles = ceil_div(T, kAttnTile);
  p.scale = scale;
  p.gate = gate; p.tab = tab; p.key_pad = key_pad;
  p.out = static_cast<__nv_bfloat16*>(out);
  p.lse = lse;
  B200_CHECK_CUDA(cudaFuncSetAttribute(attn_fwd_long_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kLfSmem));
  B200_CHECK_CUDA(launch_pdl(attn_fwd_long_kernel, dim3(ceil_div(T, 2 * kAttnTile), H, B), dim3(kLfThreads), kLfSmem,
                             static_cast<cudaStream_t>(stream), tm, p, tab_radius));
  B200_CHECK_LAUNCH();
  return 0;
}

int b200s_attn_bwd_long(const void* qkv, const void* out, const void* dout, const float* gate, const float* tab, int tab_radius,
                        const uint8_t* key_pad, const float* lse, float* delta, void* dqkv, float* dgate, float* dtab, int B,
                        int T, int H, float scale, b200s_stream stream) {
  B200_CHECK_ARG(qkv && out && dout && lse && delta && dqkv, "attn_bwd_long: null pointer");
  B200_CHECK_ARG(!tab || (dgate && dtab), "attn_bwd_long: bias given but dgate/dtab missing");
  if (int rc = check_long_shape("attn_bwd_long", B, T, H, tab_radius, tab != nullptr)) return rc;
  const int D = H * kHeadDim;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  B200_CHECK_CUDA(launch_attn_delta(out, dout, B, T, H, delta, st));
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
  const int R = tab != nullptr ? tab_radius : 0;
  dim3 grid(p.n_tiles, H, B);
  void (*kv)(const CUtensorMap, const CUtensorMap, const AttnParams, int) =
      tab != nullptr ? attn_bwd_dkv_long_kernel<true> : attn_bwd_dkv_long_kernel<false>;
  void (*dq)(const CUtensorMap, const CUtensorMap, const AttnParams, int) =
      tab != nullptr ? attn_bwd_dq_long_kernel<true> : attn_bwd_dq_long_kernel<false>;
  B200_CHECK_CUDA(cudaFuncSetAttribute(kv, cudaFuncAttributeMaxDynamicSharedMemorySize, kLkSmem));
  B200_CHECK_CUDA(launch_pdl(kv, dim3(grid), dim3(256), kLkSmem, st, tm_qkv, tm_do, p, R));
  B200_CHECK_LAUNCH();
  B200_CHECK_CUDA(cudaFuncSetAttribute(dq, cudaFuncAttributeMaxDynamicSharedMemorySize, kLqSmem));
  B200_CHECK_CUDA(launch_pdl(dq, dim3(grid), dim3(256), kLqSmem, st, tm_qkv, tm_do, p, R));
  B200_CHECK_LAUNCH();
  return 0;
}

}  // extern "C"
