// Spatial self-attention with the reference bank, head dims 64 to 128 (CLIP: d = 64; the UNet's 32x32 level: d = 80):
// flash attention with TWO 128-row query tiles per CTA processed in ping-pong.
//
//   warp 0 lane 0 : TMA      - Q tiles A and B once; K/V tiles in rings shared by both query tiles
//   warp 1 / 3    : MMA      - warp 1 drives query tile A, warp 3 tile B (whole warp + one elected lane, descriptors in
//                              uniform registers): S_X = Q_X K^T (128x128xdp) as soon as the softmax group has pulled
//                              the previous S_X into registers, O_X += P_X V (128xdpx128) when P_X is in shared memory
//   warp 2        : TMEM allocator (512 columns: S_A, S_B, O_A, O_B)
//   warps 4-7     : softmax warpgroup A (one thread per query row = TMEM lane)
//   warps 8-11    : softmax warpgroup B - started one exponential phase after A, so that one group's loads, stores and
//                              waits run under the other group's MUFU work instead of both idling the pipe together
// A softmax thread pulls its whole 128-key row of S into registers (128 of the 168 the launch bound allows) and
// releases S_X at once, so Q_X K[j+1]^T runs underneath the exponentials of tile j and
// the MUFU pipe never waits for the tensor pipe.
// Softmax: base-2 exponentials (ex2.approx), fp32 running sum, LAZY rescaling — the reference maximum of a row is only
// moved (and O rescaled in TMEM) when the tile maximum exceeds it by more than 2^8, which keeps P within fp16
// range and is exact after the final division by the row sum. P goes to shared memory as the 128B-swizzled K-major A
// operand of the P.V MMA; V tiles are used in place as MN-major B operands.
#include <cuda_runtime.h>

#include "../../include/mimo_b200.h"
#include "attn_common.h"
#include "host_util.h"
#include "ptx.cuh"

namespace mimo {

constexpr int kPPThreads = 384;
constexpr int kPPPBytes = 2 * 2 * kChunkBytes;  // P_A, P_B (two 64-key chunks each)
constexpr float kRescaleThreshold = 8.0f;       // log2 units

// NCH = 64-element chunks of the head dim (1: d <= 64, 2: d <= 128). K and V tiles live in separate rings with their
// own barriers: a K stage is released as soon as both query tiles have issued Q.K^T on it, a V stage after both P.V,
// so even single-stage rings (NCH = 2, where shared memory is tight) keep TMA one tile ahead of the tensor pipe.
template <int NCH>
struct PPCfg {
  static constexpr int kStages = NCH == 1 ? 2 : 1;
  static constexpr int kTile = NCH * kChunkBytes;  // one 128-row K or V (or Q) tile
  static constexpr int kQBytes = 2 * kTile;
  static constexpr int kSmem = kQBytes + 2 * kStages * kTile + kPPPBytes + 256;
};

__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

template <int NCH, bool kBf16>
__global__ void __launch_bounds__(kPPThreads, 1)
attn_spatial_pp_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                       const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmBK,
                       const __grid_constant__ CUtensorMap tmBV, AttnArgs a) {
  using C = Cvt<kBf16>;
  using Cfg = PPCfg<NCH>;
  constexpr int ST = Cfg::kStages;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sQ = smem;
  uint8_t* sK = sQ + Cfg::kQBytes;
  uint8_t* sV = sK + ST * Cfg::kTile;
  uint8_t* sP = sV + ST * Cfg::kTile;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sP + kPPPBytes);
  uint64_t* q_full = bars;          // 1
  uint64_t* k_full = bars + 1;      // ST (<= 2)
  uint64_t* k_empty = bars + 3;     // ST
  uint64_t* v_full = bars + 5;      // ST
  uint64_t* v_empty = bars + 7;     // ST
  uint64_t* s_full = bars + 9;      // 2 (per query tile)
  uint64_t* p_full = bars + 11;     // 2
  uint64_t* o_done = bars + 13;     // 2
  uint64_t* s_free = bars + 15;     // 2: the softmax group holds S_X in registers
  uint64_t* stagger = bars + 17;    // 1: tile A finished its first exponentials -> tile B may start (anti-phase)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 18);

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);  // provably warp-uniform for the compiler
  const int lane = threadIdx.x & 31;
  const int q_pair = blockIdx.x;
  const int h = blockIdx.y;
  const int n = blockIdx.z;
  pdl_launch_dependents();

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmV);
    tma_prefetch_desc(&tmBK);
    tma_prefetch_desc(&tmBV);
  }
  if (warp == 1 && lane == 0) {
    mbar_init(q_full, 1);
    for (int s = 0; s < ST; ++s) {
      mbar_init(&k_full[s], 1);
      mbar_init(&k_empty[s], 2);  // one tcgen05.commit per query tile
      mbar_init(&v_full[s], 1);
      mbar_init(&v_empty[s], 2);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&s_full[s], 1);
      mbar_init(&p_full[s], 4);
      mbar_init(&o_done[s], 1);
      mbar_init(&s_free[s], 4);
    }
    mbar_init(stagger, 4);
    fence_mbar_init();
  }
  if (warp == 2) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);
  // columns: S_A [0,128)  S_B [128,256)  O_A [256,384)  O_B [384,512)
  pdl_wait();  // the prologue above touched only shared memory / TMEM / kernel parameters
  const int bidx = __shfl_sync(0xffffffffu, a.bank_index ? a.bank_index[n] : -1, 0);
  const int T = a.n_self_tiles + (bidx >= 0 ? a.n_bank_tiles : 0);

  if (warp < 4) {
   if (warp == 0 && lane == 0) {
    // ===================== TMA producer =====================
    mbar_expect_tx(q_full, Cfg::kQBytes);
#pragma unroll
    for (int ch = 0; ch < NCH; ++ch) {
      tma_load_4d(sQ + ch * kChunkBytes, &tmQ, q_full, ch * 64, h, q_pair * 2 * BQ, n);
      tma_load_4d(sQ + Cfg::kTile + ch * kChunkBytes, &tmQ, q_full, ch * 64, h, q_pair * 2 * BQ + BQ, n);
    }
    for (int j = 0; j < T; ++j) {
      const int stage = j % ST;
      const uint32_t ph = ((j / ST) & 1u) ^ 1u;
      const bool bank = j >= a.n_self_tiles;
      const int row0 = (bank ? j - a.n_self_tiles : j) * BKV;
      const int img = bank ? bidx : n;
      mbar_wait(&k_empty[stage], ph);
      mbar_expect_tx(&k_full[stage], Cfg::kTile);
#pragma unroll
      for (int ch = 0; ch < NCH; ++ch)
        tma_load_4d(sK + stage * Cfg::kTile + ch * kChunkBytes, bank ? &tmBK : &tmK, &k_full[stage], ch * 64, h, row0, img);
      mbar_wait(&v_empty[stage], ph);
      mbar_expect_tx(&v_full[stage], Cfg::kTile);
#pragma unroll
      for (int ch = 0; ch < NCH; ++ch)
        tma_load_4d(sV + stage * Cfg::kTile + ch * kChunkBytes, bank ? &tmBV : &tmV, &v_full[stage], ch * 64, h, row0, img);
    }
   } else if (warp == 1 || warp == 3) {
    // ===================== MMA issuers: warp 1 drives query tile A, warp 3 tile B =====================
    // The whole warp runs the (uniform) control flow and one elected lane issues the tcgen05 instructions, so the
    // descriptors stay in uniform registers: a lane-0-only branch costs ~150 clk of scalar code per MMA here, more
    // than the MMA itself, and made the issuer the bottleneck of the kernel.
    const int x = warp == 3 ? 1 : 0;
    const uint32_t idesc_qk = make_idesc_f16(BQ, BKV, kBf16, false, false);
    const uint32_t idesc_pv = make_idesc_f16(BQ, a.dp, kBf16, false, true);  // B (= V) is MN-major
    const int ksteps_qk = a.dp / 16;
    const uint32_t qa = smem_u32(sQ) + x * Cfg::kTile;
    const uint32_t pa0 = smem_u32(sP) + x * 2 * kChunkBytes;
    const uint32_t tS = tmem_base + x * 128;
    const uint32_t tO = tmem_base + 256 + x * 128;
    auto issue_qk = [&](int j) {
      const uint32_t k_addr = smem_u32(sK + (j % ST) * Cfg::kTile);
      if (elect_one()) {
        for (int ks = 0; ks < ksteps_qk; ++ks) {
          const uint32_t off = (ks >> 2) * kChunkBytes + (ks & 3) * 32;
          umma_ss(tS, make_smem_desc_sw128(qa + off, 16, 1024), make_smem_desc_sw128(k_addr + off, 16, 1024),
                  idesc_qk, ks != 0 ? 1u : 0u);
        }
        tc_commit(&s_full[x]);
        tc_commit(&k_empty[j % ST]);  // released once both query tiles have consumed K[j]
      }
      __syncwarp();
    };
    mbar_wait(q_full, 0);
    mbar_wait(&k_full[0], 0);
    tc_fence_after();
    issue_qk(0);
    for (int j = 0; j < T; ++j) {
      const int stage = j % ST;
      if (j + 1 < T) {  // S_X(j+1) as soon as the softmax group has S_X(j) in registers
        mbar_wait(&s_free[x], j & 1);
        mbar_wait(&k_full[(j + 1) % ST], ((j + 1) / ST) & 1u);
        tc_fence_after();
        issue_qk(j + 1);
      }
      mbar_wait(&p_full[x], j & 1);
      mbar_wait(&v_full[stage], (j / ST) & 1u);
      tc_fence_after();
      const uint32_t v_addr = smem_u32(sV + stage * Cfg::kTile);
      if (elect_one()) {
#pragma unroll
        for (int ks = 0; ks < BKV / 16; ++ks) {
          const uint32_t pa = pa0 + (ks >> 2) * kChunkBytes + (ks & 3) * 32;
          umma_ss(tO, make_smem_desc_sw128(pa, 16, 1024), make_smem_desc_sw128(v_addr + ks * 2048, kChunkBytes, 1024),
                  idesc_pv, (j | ks) != 0 ? 1u : 0u);
        }
        tc_commit(&v_empty[stage]);  // released once both query tiles are done with V[j]
        tc_commit(&o_done[x]);
      }
      __syncwarp();
    }
   }
  } else {
    // ===================== softmax warpgroups =====================
    const int x = (warp - 4) >> 2;  // query tile A / B
    const int ew = warp & 3;
    const int r = ew * 32 + lane;
    const uint32_t lane_off = static_cast<uint32_t>(ew * 32) << 16;
    const uint32_t tS = tmem_base + x * 128 + lane_off;
    const uint32_t tO = tmem_base + 256 + x * 128 + lane_off;
    uint8_t* prow = sP + x * 2 * kChunkBytes + r * 128;
    const int sw = r & 7;
    const float sc = a.scale_log2;
    float m_ref = 0.f, l = 0.f;
    for (int j = 0; j < T; ++j) {
      const bool bank = j >= a.n_self_tiles;
      const int len = bank ? a.lb : a.lq;
      const int row0 = (bank ? j - a.n_self_tiles : j) * BKV;
      int valid = len - row0;
      if (valid > BKV) valid = BKV;
      mbar_wait(&s_full[x], j & 1);
      tc_fence_after();
      // ---- the whole row of S -> registers, then hand S_X back to the tensor pipe ----
      uint32_t sv[4][32];
      tmem_ld_x32(tS, sv[0]);
      tmem_ld_x32(tS + 32, sv[1]);
      tmem_ld_x32(tS + 64, sv[2]);
      tmem_ld_x32(tS + 96, sv[3]);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&s_free[x]);
      // ---- tile maximum (4 independent chains) ----
      float mx0 = -INFINITY, mx1 = -INFINITY, mx2 = -INFINITY, mx3 = -INFINITY;
      if (valid == BKV) {
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          mx0 = fmaxf(mx0, __uint_as_float(sv[0][i]));
          mx1 = fmaxf(mx1, __uint_as_float(sv[1][i]));
          mx2 = fmaxf(mx2, __uint_as_float(sv[2][i]));
          mx3 = fmaxf(mx3, __uint_as_float(sv[3][i]));
        }
      } else {
#pragma unroll
        for (int i = 0; i < 128; ++i) {
          if (i >= valid) sv[i >> 5][i & 31] = __float_as_uint(-INFINITY);  // exp2 -> 0: padded keys leave P and l
          mx0 = fmaxf(mx0, __uint_as_float(sv[i >> 5][i & 31]));
        }
      }
      const float mx = fmaxf(fmaxf(mx0, mx1), fmaxf(mx2, mx3)) * sc;
      // ---- lazy rescale decision ----
      float alpha = 1.0f;
      bool rescale = false;
      if (j == 0) {
        m_ref = mx;
      } else {
        const bool need = mx > m_ref + kRescaleThreshold;
        rescale = __any_sync(0xffffffffu, need);
        if (need) {
          alpha = fast_exp2(m_ref - mx);
          m_ref = mx;
          l *= alpha;
        }
      }
      // The two groups share one MUFU pipe per SM sub-partition. Started together they stay in lockstep - both in
      // their exponentials (each at half rate), then both in their MUFU-free part - so B is held back once, by
      // the length of A's first exponential phase, and from then on one group's loads / stores / waits hide under
      // the other's exponentials.
      if (j == 0 && x == 1) mbar_wait(stagger, 0);
      // ---- probabilities (packed in registers) ----
      float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
      const float nm = -m_ref;
      uint32_t pk[64];
#pragma unroll
      for (int c = 0; c < 4; ++c) {
#pragma unroll
        for (int i = 0; i < 16; i += 2) {
          const float p0 = fast_exp2(fmaf(__uint_as_float(sv[c][2 * i]), sc, nm));
          const float p1 = fast_exp2(fmaf(__uint_as_float(sv[c][2 * i + 1]), sc, nm));
          const float p2 = fast_exp2(fmaf(__uint_as_float(sv[c][2 * i + 2]), sc, nm));
          const float p3 = fast_exp2(fmaf(__uint_as_float(sv[c][2 * i + 3]), sc, nm));
          s0 += p0;
          s1 += p1;
          s2 += p2;
          s3 += p3;
          pk[c * 16 + i] = C::pack(p0, p1);
          pk[c * 16 + i + 1] = C::pack(p2, p3);
        }
        if (c == 3 && j == 0 && x == 0) {
          __syncwarp();
          if (lane == 0) mbar_arrive(stagger);
        }
        // P_X (and O_X) may only be overwritten once the previous P_X.V has retired
        if (c == 0 && j > 0) {
          mbar_wait(&o_done[x], (j - 1) & 1);
          tc_fence_after();
        }
        uint8_t* line = prow + (c >> 1) * kChunkBytes;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int piece = (c & 1) * 4 + q;
          *reinterpret_cast<uint4*>(line + ((piece ^ sw) << 4)) =
              make_uint4(pk[c * 16 + 4 * q], pk[c * 16 + 4 * q + 1], pk[c * 16 + 4 * q + 2], pk[c * 16 + 4 * q + 3]);
        }
      }
      l += (s0 + s1) + (s2 + s3);
      // ---- correction of O (rare) ----
      if (rescale) {
        for (int c = 0; c < a.dp / 16; ++c) {
          uint32_t v[16];
          tmem_ld_x16(tO + c * 16, v);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = __float_as_uint(__uint_as_float(v[i]) * alpha);
          tmem_st_x16(tO + c * 16, v);
        }
        tmem_st_wait();
      }
      fence_proxy_async_smem();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&p_full[x]);
    }
    // ---- epilogue: O / l -> global ----
    mbar_wait(&o_done[x], (T - 1) & 1);
    tc_fence_after();
    const float inv_l = 1.0f / l;
    const int qrow = q_pair * 2 * BQ + x * BQ + r;
    typename C::T* orow =
        static_cast<typename C::T*>(a.out) + (static_cast<long long>(n) * a.lq + qrow) * a.ld_out + h * a.d;
    for (int c = 0; c < a.dp / 16; ++c) {
      uint32_t v[16];
      tmem_ld_x16(tO + c * 16, v);
      tmem_ld_wait();
      if (qrow < a.lq) {
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          if (c * 16 + q * 8 < a.d) {
            uint4 o;
            o.x = C::pack(__uint_as_float(v[q * 8 + 0]) * inv_l, __uint_as_float(v[q * 8 + 1]) * inv_l);
            o.y = C::pack(__uint_as_float(v[q * 8 + 2]) * inv_l, __uint_as_float(v[q * 8 + 3]) * inv_l);
            o.z = C::pack(__uint_as_float(v[q * 8 + 4]) * inv_l, __uint_as_float(v[q * 8 + 5]) * inv_l);
            o.w = C::pack(__uint_as_float(v[q * 8 + 6]) * inv_l, __uint_as_float(v[q * 8 + 7]) * inv_l);
            *reinterpret_cast<uint4*>(orow + c * 16 + q * 8) = o;
          }
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

template <int NCH, bool kBf16>
static int launch_pp(const CUtensorMap& q, const CUtensorMap& k, const CUtensorMap& v, const CUtensorMap& bk,
                     const CUtensorMap& bv, const AttnArgs& a, int n, cudaStream_t st) {
  using Cfg = PPCfg<NCH>;
  auto kern = attn_spatial_pp_kernel<NCH, kBf16>;
  static bool attr_done = false;
  if (!attr_done) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmem);
    if (e != cudaSuccess) return set_cuda_error("cudaFuncSetAttribute(attn_pp)", e);
    attr_done = true;
  }
  dim3 grid((a.lq + 2 * BQ - 1) / (2 * BQ), a.heads, n);
  cudaError_t e = launch_k(kern, grid, dim3(kPPThreads), Cfg::kSmem, st, q, k, v, bk, bv, a);
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) return set_cuda_error("attn_pp launch", e);
  return MIMO_OK;
}

int launch_attn_pp(bool bf16, const CUtensorMap& q, const CUtensorMap& k, const CUtensorMap& v, const CUtensorMap& bk,
                   const CUtensorMap& bv, const AttnArgs& a, int n, cudaStream_t st) {
  if (a.dp <= 64) return bf16 ? launch_pp<1, true>(q, k, v, bk, bv, a, n, st) : launch_pp<1, false>(q, k, v, bk, bv, a, n, st);
  return bf16 ? launch_pp<2, true>(q, k, v, bk, bv, a, n, st) : launch_pp<2, false>(q, k, v, bk, bv, a, n, st);
}

}  // namespace mimo
