// Flash-style attention forward with the WavLM gated relative-position bias, tcgen05 + TMEM + TMA (sm_100a).
//
// One CTA = 256 query rows of one (batch, head): two softmax warpgroups (WG) of 128 threads, each owning one 128-row query
// tile, one TMA producer warp and one MMA-issuing warp.  Thread r of a WG owns query row r (TMEM lane r): the row reference /
// sum of the softmax are thread-local, no shuffles.  Both WGs share every K/V tile (one TMA load feeds both).
// Per WG and key tile n (128 keys):
//   S_n  = Q K_n^T           tcgen05.mma 128x128x64  -> TMEM (128 columns)
//   p    = exp2(S*scale*log2e + gate_i*log2e*tab[j-i] + keymask - m_i)      ONE pass over the scores
//   P_n -> shared memory in the K-major SWIZZLE_128B operand layout (bf16)
//   O   += P_n V_n           tcgen05.mma 128x64x128 ACCUMULATING IN TMEM over the whole key loop (V_n read MN-major from the TMA tile)
// The softmax is invariant to the reference m_i subtracted in the exponent, so m_i is fixed by the first tile that has a finite
// score for the row and never refreshed: the accumulator needs no per-tile rescale and never leaves TMEM until the epilogue
// (fp32 sums / accumulators absorb factors up to 2^80).  If a later score outgrows the reference by more than that, the warp
// re-bases: it rescales its 32 accumulator rows in TMEM (tcgen05.ld / st) and recomputes the tile -- a correctness path that
// real inputs do not take.
// The MMA warp issues, per (tile, WG) in a fixed alternating order, S(n+1) and then PV(n) as soon as that WG's P_n is staged:
// the next scores are ready ~one MMA later, and the tensor core runs under the other WG's exponentials.
// Padding: key tiles that are fully padded at the END of the utterance are skipped (the loop runs over n_eff tiles), and a CTA
// whose 256 query rows are all padded only writes zeros -- padded frames never influence valid ones (keys are masked) and the
// reference's values there are unspecified garbage, so the ragged batch does not pay for its padding.
// The per-head Toeplitz bias table is kept in shared memory as FOUR copies shifted by 0..3 elements, so the 32 consecutive
// entries a thread needs per 32-column chunk are 8 aligned 128-bit loads instead of 32 scalar ones.
#include "../../include/unispeech_b200.h"
#include "attn_common.cuh"
#include "common.h"
#include <type_traits>

namespace b200 {

__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// 32 x 32 bit-matrix transpose across a warp: on entry bit j of lane l's word is element (l, j); on return bit l of lane j's
// word is that element.  Five butterfly stages (one shuffle + three logic ops each) replace 32 ballots.
__device__ __forceinline__ uint32_t warp_bit_transpose(uint32_t x, int lane) {
#pragma unroll
  for (int s = 16; s >= 1; s >>= 1) {
    const uint32_t m = (s == 16) ? 0x0000FFFFu : (s == 8) ? 0x00FF00FFu : (s == 4) ? 0x0F0F0F0Fu : (s == 2) ? 0x33333333u : 0x55555555u;
    const uint32_t y = __shfl_xor_sync(0xffffffffu, x, s);
    x = (lane & s) ? ((x & ~m) | ((y >> s) & m)) : ((x & m) | ((y << s) & ~m));
  }
  return x;
}
__device__ __forceinline__ void mbar_arrive_rel(uint64_t* bar) {
  asm volatile("mbarrier.arrive.release.cta.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// registers -> 32 lanes x 32 consecutive fp32 TMEM columns (inverse of tmem_ld_32x32b_x32)
__device__ __forceinline__ void tmem_st_32x32b_x32(uint32_t taddr, const uint32_t* r) {
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
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

constexpr int kFwdQ = 0;                   // 2 x 16 KB (one Q tile per warpgroup)
constexpr int kFwdK = 32768;               // 2 stages x 16 KB
constexpr int kFwdV = 65536;               // 2 stages x 16 KB
constexpr int kFwdP = 98304;               // 2 x 32 KB (one P tile per warpgroup)
constexpr int kFwdTab = 163840;            // fp32 bias-table copies, key mask, tile flags
constexpr int kFwdThreads = 320;           // 2 softmax warpgroups + TMA warp + MMA warp
constexpr int kTabCopies = 4;
constexpr float kRebase = 1.2089258e24f;   // 2^80: a tile whose row sum reaches this is re-based on its own maximum

// floats of ONE bias-table copy: (N + 2) * 128 entries + 8 so that consecutive copies start 8 banks apart (conflict-free
// 128-bit loads across the quarter warp, whose lanes alternate between the four copies)
__host__ __device__ constexpr int fwd_tab_stride(int N) { return (N + 2) * kAttnTile + 8; }
// dynamic shared memory of attn_fwd_kernel for N key tiles: table copies (with the bias), key mask, tile flags
constexpr int fwd_smem_bytes(int N, bool has_bias) {
  return kFwdTab + static_cast<int>(sizeof(float)) * ((has_bias ? kTabCopies * fwd_tab_stride(N) : 0) + N * kAttnTile) +
         static_cast<int>(sizeof(int)) * N + 1024;
}
constexpr int kFwdSmemMax = 232448 - 1024;

template <bool HAS_BIAS, bool DROP>
__global__ void __launch_bounds__(kFwdThreads, 1) attn_fwd_kernel(const __grid_constant__ CUtensorMap tm,
                                                                 const __grid_constant__ AttnParams p) {
  pdl_grid_sync();
  const int tid = threadIdx.x, warp = tid >> 5;
  const int wg = warp >> 2;  // 0, 1 = softmax warpgroups; 2 = TMA warp (8) and MMA warp (9)
  const int q0 = blockIdx.x * 2 * kAttnTile, h = blockIdx.y, b = blockIdx.z;
  const int T = p.T, D = p.D, N = p.n_tiles;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);  // 1024-aligned, still a __shared__ pointer (LDS/STS, not generic)
  uint8_t* sQ = smem + kFwdQ;
  uint8_t* sK = smem + kFwdK;
  uint8_t* sV = smem + kFwdV;
  uint8_t* sP = smem + kFwdP;
  float* tab_s = reinterpret_cast<float*>(smem + kFwdTab);           // [4][fwd_tab_stride(N)]: copy c holds slice[i + c]
  const int tab_stride = fwd_tab_stride(N);
  float* kbias = tab_s + (HAS_BIAS ? kTabCopies * tab_stride : 0);  // [N*128]
  int* tile_flags = reinterpret_cast<int*>(kbias + N * kAttnTile);  // [N]: 0 no masked key, 1 some, 2 all

  __shared__ uint64_t q_full, k_full[2], k_empty[2], v_full[2], v_empty[2], s_full[2], p_ready[2], pv_done[2];
  __shared__ uint32_t tmem_base_s;

  // ---- key padding: additive mask, per-tile flags, number of key tiles that hold any valid key, and whether any of this CTA's
  // 256 query rows is live.  ONE pass over the utterance's pad bytes (every thread takes a few), shared-memory counters, one
  // barrier: the prologue pays a single global-load latency instead of one per key tile.
  __shared__ int n_eff_s, live_s;
  for (int t = tid; t < N; t += kFwdThreads) tile_flags[t] = 0;   // masked keys per tile (turned into 0 / 1 / 2 below)
  if (tid == 0) { n_eff_s = 1; live_s = 0; }
  __syncthreads();
  {
    int last_valid = -1;
    bool live = false;
    for (int j = tid; j < N * kAttnTile; j += kFwdThreads) {
      const bool masked = (j >= T) || (p.key_pad != nullptr && p.key_pad[static_cast<long long>(b) * T + j] != 0);
      kbias[j] = masked ? -INFINITY : 0.f;
      if (masked) atomicAdd(&tile_flags[j / kAttnTile], 1);
      else last_valid = j;                                     // increasing j: the last hit is the largest
      if (!masked && j >= q0 && j < q0 + 2 * kAttnTile) live = true;
    }
    if (last_valid >= 0) atomicMax(&n_eff_s, last_valid / kAttnTile + 1);
    if (live) live_s = 1;
  }
  __syncthreads();
  const int n_eff = n_eff_s;
  // ---- a CTA whose query rows are all padded (or beyond T) has nothing to compute
  if (p.key_pad != nullptr && live_s == 0) {
    if (tid < 2 * kAttnTile && q0 + tid < T) {
      uint4* dst = reinterpret_cast<uint4*>(p.out + (static_cast<long long>(b) * T + q0 + tid) * D + h * kHeadDim);
#pragma unroll
      for (int g = 0; g < 8; ++g) dst[g] = make_uint4(0u, 0u, 0u, 0u);
      if (p.lse != nullptr) p.lse[(static_cast<long long>(b) * p.H + h) * T + q0 + tid] = INFINITY;
    }
    return;
  }
  for (int t = tid; t < N; t += kFwdThreads) {  // counts -> 0 no masked key, 1 some, 2 all (read after the barrier below)
    const int c = tile_flags[t];
    tile_flags[t] = (c == 0) ? 0 : (c == kAttnTile ? 2 : 1);
  }

  if (warp == 8 && (tid & 31) == 0) {
    // the TMA thread initialises the barriers itself and puts Q and the first K / V tiles in flight right away: they land while
    // the rest of the CTA is still filling the bias-table copies (the other warps see the barriers after the __syncthreads below)
    tma_prefetch_desc(&tm);
    mbar_init(&q_full, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&k_full[i], 1);
      mbar_init(&v_full[i], 1);
      mbar_init(&k_empty[i], 1);   // tcgen05.commit after the second warpgroup's S MMA
      mbar_init(&v_empty[i], 1);   // ... after the second warpgroup's PV MMA
      mbar_init(&s_full[i], 1);    // index = warpgroup
      mbar_init(&pv_done[i], 1);
      mbar_init(&p_ready[i], kAttnTile);
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
  if (HAS_BIAS) {
    const int len = (N + 2) * kAttnTile;
    const int base = (T - 1) - (q0 + 2 * kAttnTile - 1);
    const float* tab_h = p.tab + static_cast<long long>(h) * (2 * T - 1);
    for (int i = tid; i < kTabCopies * len; i += kFwdThreads) {
      const int c = i / len, k = i - c * len;
      const int gi = k + c + base;
      tab_s[c * tab_stride + k] = (gi >= 0 && gi < 2 * T - 1) ? tab_h[gi] : 0.f;
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;

  if (warp == 8) {
    // ------------------------------------------------------------------ TMA producer warp
    if ((tid & 31) == 0) {
      for (int n = 1; n < n_eff; ++n) {  // (Q and tile 0 were issued in the prologue)
        const int s = n & 1;
        const uint32_t ph = (n >> 1) & 1;
        mbar_wait(&k_empty[s], ph ^ 1);
        mbar_expect_tx(&k_full[s], 16384);
        tma_load_4d(sK + s * 16384, &tm, &k_full[s], D + h * kHeadDim, n * kAttnTile, b, 0);
        mbar_wait(&v_empty[s], ph ^ 1);
        mbar_expect_tx(&v_full[s], 16384);
        tma_load_4d(sV + s * 16384, &tm, &v_full[s], 2 * D + h * kHeadDim, n * kAttnTile, b, 0);
      }
    }
  } else if (warp == 9) {
    // ------------------------------------------------------------------ MMA-issuing warp (one thread)
    if ((tid & 31) == 0) {
      constexpr uint32_t idesc_s = make_idesc_bf16(128, 128, 0, 0);
      constexpr uint32_t idesc_pv = make_idesc_bf16(128, 64, 0, 1);
      auto issue_s = [&](int w, int n) {  // S_n of warpgroup w
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
          mbar_wait(&p_ready[w], n & 1);  // P_n of this warpgroup is staged and its S_n has been read
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
    const int r = tid & 127;                 // row inside this warpgroup's tile == TMEM lane
    const int r256 = wg * kAttnTile + r;     // row inside the CTA's 256-row block
    const int lane = tid & 31;
    const bool row_valid = (q0 + r256) < T;
    const uint32_t lane_addr = static_cast<uint32_t>((warp & 3) * 32) << 16;
    const uint32_t s_addr = tmem + wg * 256 + lane_addr;        // S: 128 columns
    const uint32_t o_addr = tmem + wg * 256 + 128 + lane_addr;  // O: 64 columns
    uint8_t* sPw = sP + wg * 32768;

    float gl = 0.f;
    if (HAS_BIAS) {
      const float g = (p.gate != nullptr && row_valid) ? p.gate[(static_cast<long long>(b) * p.H + h) * T + q0 + r256] : 1.0f;
      gl = g * kLog2e;
    }
    const float sc = p.scale * kLog2e;
    // this row's window of the bias table: entry (key j) = slice[j + 255 - r256]; copy a = (255 - r256) & 3 is the one in which
    // that window starts on a 16-byte boundary
    const int toff = 2 * kAttnTile - 1 - r256;
    const float4* tab4 = reinterpret_cast<const float4*>(tab_s + (toff & 3) * tab_stride + (toff & ~3));
    // dropout on the probabilities: per-row hash keys, and where this warp's 32 rows keep their bits (one word per key column)
    uint32_t rk0 = 0, rk1 = 0;
    uint32_t* mask_row = nullptr;
    if (DROP) {
      const uint32_t rowid = static_cast<uint32_t>(b * p.H + h) * static_cast<uint32_t>(T) + static_cast<uint32_t>(q0 + r256);
      rk0 = drop_row_k0(p.drop_k0, rowid);
      rk1 = drop_row_k1(p.drop_k1, rowid);
      if (q0 + wg * kAttnTile < N * kAttnTile)  // (a 256-row CTA may reach past the last 128-row tile: nothing to record there)
        mask_row = p.drop_mask + (static_cast<long long>(b * p.H + h) * (4 * N) + ((q0 + r256) >> 5)) * (N * kAttnTile);
    }

    float m_ref = -INFINITY, l_run = 0.f;

    for (int n = 0; n < n_eff; ++n) {
      const int k0 = n * kAttnTile;
      mbar_wait(&s_full[wg], n & 1);
      tc_fence_after();
      const bool msk = tile_flags[n] != 0;

      auto tile_max = [&]() {  // row maximum of the exponent argument over this tile (bias and key mask included)
        float mx = -INFINITY;
#pragma unroll 1
        for (int c0 = 0; c0 < kAttnTile; c0 += 32) {
          uint32_t su[32];
          tmem_ld_32x32b_x32(s_addr + c0, su);
          tmem_ld_wait();
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            float4 tb = make_float4(0.f, 0.f, 0.f, 0.f);
            if (HAS_BIAS) tb = tab4[(k0 + c0) / 4 + q];
            float x0 = __uint_as_float(su[4 * q]) * sc, x1 = __uint_as_float(su[4 * q + 1]) * sc;
            float x2 = __uint_as_float(su[4 * q + 2]) * sc, x3 = __uint_as_float(su[4 * q + 3]) * sc;
            if (HAS_BIAS) {
              x0 = fmaf(gl, tb.x, x0); x1 = fmaf(gl, tb.y, x1); x2 = fmaf(gl, tb.z, x2); x3 = fmaf(gl, tb.w, x3);
            }
            if (msk) {
              const float4 kb = *reinterpret_cast<const float4*>(kbias + k0 + c0 + 4 * q);
              x0 += kb.x; x1 += kb.y; x2 += kb.z; x3 += kb.w;
            }
            mx = fmaxf(fmaxf(mx, fmaxf(x0, x1)), fmaxf(x2, x3));
          }
        }
        return mx;
      };

      // rows that have not seen a finite score yet take this tile's maximum as their reference (first tile, or only masked
      // keys so far); they hold l = 0 and an all-zero accumulator, so nothing has to be rescaled
      if (__any_sync(0xffffffffu, m_ref == -INFINITY)) {
        const float mx = tile_max();
        if (m_ref == -INFINITY) m_ref = mx;
      }
      bool p_free = (n == 0);  // PV(n-1) must have consumed the P buffer before it is overwritten
      // one pass over the tile: probabilities (relative to m_ref) -> bf16 P tile in shared memory; returns the row sum.
      // MSK is a compile-time flag so that the common tiles (no padded key) carry no mask arithmetic at all.
      auto softmax_tile = [&](auto MSK) -> float {
        constexpr bool kMsk = decltype(MSK)::value;
        const float neg_ref = (m_ref == -INFINITY) ? 0.f : -m_ref;
        float part0 = 0.f, part1 = 0.f, part2 = 0.f, part3 = 0.f;
        uint32_t sa[32], sb[32];
        tmem_ld_32x32b_x32(s_addr, sa);
        tmem_ld_wait();
#pragma unroll
        for (int cc = 0; cc < 4; ++cc) {
          const int c0 = cc * 32;
          uint32_t* su = (cc & 1) ? sb : sa;
          if (cc + 1 < 4) tmem_ld_32x32b_x32(s_addr + c0 + 32, (cc & 1) ? sa : sb);  // next chunk in flight under this one
          float pv[32];
          uint32_t rowbits = 0, hbits = 0;
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            float4 tb = make_float4(0.f, 0.f, 0.f, 0.f), kb = make_float4(0.f, 0.f, 0.f, 0.f);
            if (HAS_BIAS) tb = tab4[(k0 + c0) / 4 + q];
            if (kMsk) kb = *reinterpret_cast<const float4*>(kbias + k0 + c0 + 4 * q);
            const float tbv[4] = {tb.x, tb.y, tb.z, tb.w};
            const float kbv[4] = {kb.x, kb.y, kb.z, kb.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const int j = 4 * q + e;
              float x = fmaf(__uint_as_float(su[j]), sc, neg_ref);
              if (HAS_BIAS) x = fmaf(gl, tbv[e], x);
              if (kMsk) x += kbv[e];
              const float ex = fast_exp2(x);
              // four independent partial sums: the normaliser (taken before dropout) is not one 128-long dependent chain
              if (e == 0) part0 += ex; else if (e == 1) part1 += ex; else if (e == 2) part2 += ex; else part3 += ex;
              if (DROP) {
                if ((j & 1) == 0) hbits = drop_bits(rk0, rk1, static_cast<uint32_t>(k0 + c0 + j) >> 1);
                const bool keep = (j & 1) ? drop_keep_hi(hbits, p.drop_thr_hi) : drop_keep_lo(hbits, p.drop_thr_hi);
                if (keep) rowbits |= (1u << j);  // this row's decisions for the 32 key columns
                pv[j] = keep ? ex : 0.f;
              } else {
                pv[j] = ex;
              }
            }
          }
          if (DROP) {
            // the backward walks key-major: store, per key column, one word whose bit l is the decision of query row l of this warp
            const uint32_t mword = warp_bit_transpose(rowbits, lane);
            if (mask_row != nullptr) mask_row[k0 + c0 + lane] = mword;
          }
          if (!p_free) {
            mbar_wait(&pv_done[wg], (n - 1) & 1);
            p_free = true;
          }
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            uint4 w;
            w.x = pack_bf16x2(pv[g * 8 + 0], pv[g * 8 + 1]);
            w.y = pack_bf16x2(pv[g * 8 + 2], pv[g * 8 + 3]);
            w.z = pack_bf16x2(pv[g * 8 + 4], pv[g * 8 + 5]);
            w.w = pack_bf16x2(pv[g * 8 + 6], pv[g * 8 + 7]);
            store_sw128_chunk(sPw, r, (c0 >> 3) + g, w);
          }
          if (cc + 1 < 4) tmem_ld_wait();
        }
        return (part0 + part1) + (part2 + part3);
      };
      float lsum;
#pragma unroll 1
      while (true) {
        lsum = msk ? softmax_tile(std::true_type{}) : softmax_tile(std::false_type{});
        if (!__any_sync(0xffffffffu, !(lsum < kRebase))) break;
        // ---- re-base (rare): a score outgrew the reference by 2^80.  Move this warp's rows to the tile maximum: rescale the row
        // sums and the accumulator rows in TMEM (all PV MMAs issued so far have retired once pv_done(n-1) fired; PV(n) cannot
        // be issued before this warpgroup arrives on p_ready), then recompute the tile.
        const float m_new = fmaxf(m_ref, tile_max());
        const float factor = (m_ref == -INFINITY) ? 0.f : fast_exp2(m_ref - m_new);
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
            tmem_st_32x32b_x32(o_addr + hlf * 32, t0);
          }
          tmem_st_wait();
        }
        l_run *= factor;
        m_ref = m_new;
      }
      l_run += lsum;

      fence_proxy_async_smem();  // generic-proxy smem writes -> visible to the tensor core (async proxy)
      tc_fence_before();
      mbar_arrive_rel(&p_ready[wg]);
    }
    mbar_wait(&pv_done[wg], (n_eff - 1) & 1);
    tc_fence_after();

    uint32_t t0[32], t1[32];
    tmem_ld_32x32b_x32(o_addr, t0);
    tmem_ld_32x32b_x32(o_addr + 32, t1);
    tmem_ld_wait();
    if (row_valid) {
      const float inv = l_run > 0.f ? (DROP ? p.drop_rp : 1.0f) / l_run : 0.f;
      __nv_bfloat16* dst = p.out + (static_cast<long long>(b) * T + q0 + r256) * D + h * kHeadDim;
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        uint4 w;
        w.x = pack_bf16x2(__uint_as_float(t0[g * 8 + 0]) * inv, __uint_as_float(t0[g * 8 + 1]) * inv);
        w.y = pack_bf16x2(__uint_as_float(t0[g * 8 + 2]) * inv, __uint_as_float(t0[g * 8 + 3]) * inv);
        w.z = pack_bf16x2(__uint_as_float(t0[g * 8 + 4]) * inv, __uint_as_float(t0[g * 8 + 5]) * inv);
        w.w = pack_bf16x2(__uint_as_float(t0[g * 8 + 6]) * inv, __uint_as_float(t0[g * 8 + 7]) * inv);
        *reinterpret_cast<uint4*>(dst + g * 8) = w;
      }
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        uint4 w;
        w.x = pack_bf16x2(__uint_as_float(t1[g * 8 + 0]) * inv, __uint_as_float(t1[g * 8 + 1]) * inv);
        w.y = pack_bf16x2(__uint_as_float(t1[g * 8 + 2]) * inv, __uint_as_float(t1[g * 8 + 3]) * inv);
        w.z = pack_bf16x2(__uint_as_float(t1[g * 8 + 4]) * inv, __uint_as_float(t1[g * 8 + 5]) * inv);
        w.w = pack_bf16x2(__uint_as_float(t1[g * 8 + 6]) * inv, __uint_as_float(t1[g * 8 + 7]) * inv);
        *reinterpret_cast<uint4*>(dst + 32 + g * 8) = w;
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

int make_qkv_tmap(CUtensorMap* out, const void* qkv, int T, int B, int D3, int box_rows);

}  // namespace b200

using namespace b200;

extern "C" {

// out[b,t,h*64+d] = softmax_j(scale q.k + gate*tab[j-i], key padding) v     (WavLM/modules.py:540-563 replaced)
// qkv: bf16 [B,T,3D] fused projection output; gate: fp32 [B,H,T] or NULL; tab: fp32 [H,2T-1] or NULL (no bias);
// key_pad: uint8 [B,T] or NULL; out: bf16 [B,T,D]; lse: fp32 [B,H,T] (log2-domain log-sum-exp, saved for backward).
// Rows of `out` at padded query frames are unspecified-but-finite (zeros where a whole 256-row block is padded).
int b200s_attn_fwd_dropout(const void* qkv, const float* gate, const float* tab, const uint8_t* key_pad, void* out, float* lse,
                           int B, int T, int H, float scale, float drop_p, uint32_t key0, uint32_t key1, uint32_t* drop_mask,
                           b200s_stream stream) {
  B200_CHECK_ARG(qkv && out, "attn_fwd: null pointer");
  B200_CHECK_ARG(drop_p >= 0.f && drop_p < 1.f, "attn_fwd: dropout p=%f out of range [0,1)", static_cast<double>(drop_p));
  B200_CHECK_ARG(drop_p == 0.f || drop_mask != nullptr, "attn_fwd: dropout needs the mask buffer (b200s_attn_dropout_mask_words)");
  B200_CHECK_ARG(static_cast<long long>(B) * H * T < (1LL << 32), "attn_fwd: B*H*T exceeds the 32-bit dropout row counter");
  const int D = H * kHeadDim;
  CUtensorMap tm;
  AttnParams p;
  memset(&p, 0, sizeof(p));
  p.T = T; p.H = H; p.B = B; p.D = D;
  p.n_tiles = ceil_div(T, kAttnTile);
  const int smem = fwd_smem_bytes(p.n_tiles, tab != nullptr);
  B200_CHECK_ARG(T >= 1 && smem <= kFwdSmemMax, "attn_fwd: T=%d out of range (needs %d bytes of shared memory)", T, smem);
  if (make_qkv_tmap(&tm, qkv, T, B, 3 * D, kAttnTile)) return -3;
  p.scale = scale;
  p.gate = gate; p.tab = tab; p.key_pad = key_pad;
  p.out = static_cast<__nv_bfloat16*>(out);
  p.lse = lse;
  const bool drop = drop_p > 0.f;
  p.drop_mask = drop_mask;
  p.drop_k0 = key0; p.drop_k1 = key1;
  p.drop_thr_hi = drop_threshold16(drop_p) << 16;
  p.drop_rp = 1.0f / (1.0f - drop_p);
  dim3 grid(ceil_div(T, 2 * kAttnTile), H, B);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  void (*kern)(const CUtensorMap, const AttnParams) =
      tab != nullptr ? (drop ? attn_fwd_kernel<true, true> : attn_fwd_kernel<true, false>)
                     : (drop ? attn_fwd_kernel<false, true> : attn_fwd_kernel<false, false>);
  B200_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  B200_CHECK_CUDA(launch_pdl(kern, dim3(grid), dim3(kFwdThreads), smem, st, tm, p));
  B200_CHECK_LAUNCH();
  return 0;
}

int b200s_attn_fwd(const void* qkv, const float* gate, const float* tab, const uint8_t* key_pad, void* out, float* lse,
                   int B, int T, int H, float scale, b200s_stream stream) {
  return b200s_attn_fwd_dropout(qkv, gate, tab, key_pad, out, lse, B, T, H, scale, 0.f, 0u, 0u, nullptr, stream);
}

long long b200s_attn_dropout_mask_words(int B, int T, int H) { return attn_drop_mask_words(B, H, T); }

int b200s_attn_fwd_max_frames(int has_bias) {
  int n = 1;
  while (fwd_smem_bytes(n + 1, has_bias != 0) <= kFwdSmemMax) ++n;
  return n * kAttnTile;
}

}  // extern "C"
