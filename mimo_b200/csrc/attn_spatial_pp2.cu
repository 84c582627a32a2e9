// Spatial self-attention with the reference bank, head dims with d + 1 <= 64 (the UNet's 64x64 level: d = 40): the
// ping-pong flash attention of attn_spatial_pp.cu with TWO softmax threads per query row and the row sum computed by
// the tensor pipe.
//
// Why: at d = 40 the kernel is bound by the MUFU pipe (16 ex2 / clk / SM). With one thread per row (128 S values in
// registers, 8 softmax warps) every SM sub-partition hosts two softmax warps whose exponential phases and MUFU-free phases
// (TMEM load, row maximum, pack, shared-memory stores, barrier waits) alternate - measured 64 % MUFU utilisation. Here a
// row is split between two threads of two different warps (64 S values each, 16 softmax warps, four per sub-partition),
// so some warp always has exponentials to issue, and three per-element instructions disappear:
//   * the running row sum: V gets a column of ones (written into the landed V tile at channel d, which TMA zero-filled),
//     so O[:, d] accumulates sum_k P[q, k] of exactly the fp16-rounded P that multiplies V - no FADD per element, no
//     cross-thread sum, and lazy rescaling treats it like any other O column;
//   * P is packed and stored 16 values at a time straight out of the S registers (no second register array).
// Measured on B200 (profiles/r02_attn_ab*.log, n = 48, 4096 queries, 8192 / 4096 keys, d = 40): 3.34 ms vs 3.62 ms for the
// one-thread-per-row kernel. Also tried here and dropped: a degree-4 polynomial exp2 on the FMA pipe for a quarter of the
// elements (3.48 ms: with the MUFU work already spread over 16 warps the kernel is issue-bound, the extra 8 instructions
// per offloaded element cost more than the MUFU slots they free), and ex2.approx.f16x2 (two MUFU.EX2.F16 in SASS).
//
//   warp 0        : TMA   - Q tiles A and B once; K / V tiles in rings shared by both query tiles
//   warp 1 / 3    : MMA   - warp 1 drives query tile A, warp 3 tile B (whole warp + one elected lane)
//   warp 2        : TMEM allocator (512 columns: S_A, S_B, O_A, O_B)
//   warps 4-19    : softmax group g = (warp - 4) / 4: query tile x = g / 2, key half hf = g % 2 (keys [64 hf, 64 hf + 64)
//                   of every 128-key tile); thread = TMEM lane = query row. The two halves of a row agree on the row
//                   maximum through shared memory + a 64-thread named barrier once per tile.
#include <cuda_runtime.h>

#include "../../include/mimo_b200.h"
#include "attn_common.h"
#include "host_util.h"
#include "ptx.cuh"

namespace mimo {

constexpr int kPP2Threads = 640;
constexpr int kPP2PBytes = 2 * 2 * kChunkBytes;  // P_A, P_B (two 64-key chunks each)
constexpr int kPP2MaxBytes = 2 * 2 * 2 * 128 * 4;  // [tile parity][query tile][half][row] floats
constexpr float kRescaleThreshold2 = 8.0f;       // log2 units

template <int NCH>
struct PP2Cfg {
  static constexpr int kStages = NCH == 1 ? 2 : 1;
  static constexpr int kTile = NCH * kChunkBytes;
  static constexpr int kQBytes = 2 * kTile;
  static constexpr int kSmem = kQBytes + 2 * kStages * kTile + kPP2PBytes + kPP2MaxBytes + 256;
};

__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

template <int NCH, bool kBf16>
__global__ void __launch_bounds__(kPP2Threads, 1)
attn_spatial_pp2_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                        const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmBK,
                        const __grid_constant__ CUtensorMap tmBV, AttnArgs a) {
  using C = Cvt<kBf16>;
  using Cfg = PP2Cfg<NCH>;
  constexpr int ST = Cfg::kStages;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sQ = smem;
  uint8_t* sK = sQ + Cfg::kQBytes;
  uint8_t* sV = sK + ST * Cfg::kTile;
  uint8_t* sP = sV + ST * Cfg::kTile;
  float* sMax = reinterpret_cast<float*>(sP + kPP2PBytes);
  uint64_t* bars = reinterpret_cast<uint64_t*>(sP + kPP2PBytes + kPP2MaxBytes);
  uint64_t* q_full = bars;          // 1
  uint64_t* k_full = bars + 1;      // ST (<= 2)
  uint64_t* k_empty = bars + 3;     // ST
  uint64_t* v_full = bars + 5;      // ST
  uint64_t* v_empty = bars + 7;     // ST
  uint64_t* s_full = bars + 9;      // 2 (per query tile)
  uint64_t* p_full = bars + 11;     // 2
  uint64_t* o_done = bars + 13;     // 2
  uint64_t* s_free = bars + 15;     // 2
  uint64_t* stagger = bars + 17;    // 1
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 18);

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  const int q_pair = blockIdx.x;
  const int h = blockIdx.y;
  const int n = blockIdx.z;
  pdl_launch_dependents();
  const int dpv = (a.d + 1 + 15) / 16 * 16;  // O columns: d value channels + the ones column, rounded to the MMA's N step

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
      mbar_init(&k_empty[s], 2);
      mbar_init(&v_full[s], 1);
      mbar_init(&v_empty[s], 2);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&s_full[s], 1);
      mbar_init(&p_full[s], 8);
      mbar_init(&o_done[s], 1);
      mbar_init(&s_free[s], 8);
    }
    mbar_init(stagger, 8);
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
      const int x = warp == 3 ? 1 : 0;
      const uint32_t idesc_qk = make_idesc_f16(BQ, BKV, kBf16, false, false);
      const uint32_t idesc_pv = make_idesc_f16(BQ, dpv, kBf16, false, true);  // B (= V | ones) is MN-major
      const int ksteps_qk = a.dp / 16;
      const uint32_t qa = smem_u32(sQ) + x * Cfg::kTile;
      const uint32_t pa0 = smem_u32(sP) + x * 2 * kChunkBytes;
      const uint32_t tS = tmem_base + x * 128;
      const uint32_t tO = tmem_base + 256 + x * 128;
      // the ones column: channel d of every key row of the landed V tile (128B-swizzled rows of 64 channels)
      const int one_chunk = a.d >> 6, one_ch = a.d & 63;
      const uint16_t one_bits = kBf16 ? 0x3f80 : 0x3c00;
      auto issue_qk = [&](int j) {
        const uint32_t k_addr = smem_u32(sK + (j % ST) * Cfg::kTile);
        if (elect_one()) {
          for (int ks = 0; ks < ksteps_qk; ++ks) {
            const uint32_t off = (ks >> 2) * kChunkBytes + (ks & 3) * 32;
            umma_ss(tS, make_smem_desc_sw128(qa + off, 16, 1024), make_smem_desc_sw128(k_addr + off, 16, 1024),
                    idesc_qk, ks != 0 ? 1u : 0u);
          }
          tc_commit(&s_full[x]);
          tc_commit(&k_empty[j % ST]);
        }
        __syncwarp();
      };
      mbar_wait(q_full, 0);
      mbar_wait(&k_full[0], 0);
      tc_fence_after();
      issue_qk(0);
      for (int j = 0; j < T; ++j) {
        const int stage = j % ST;
        if (j + 1 < T) {
          mbar_wait(&s_free[x], j & 1);
          mbar_wait(&k_full[(j + 1) % ST], ((j + 1) / ST) & 1u);
          tc_fence_after();
          issue_qk(j + 1);
        }
        mbar_wait(&v_full[stage], (j / ST) & 1u);
        {
          // both issuer warps write the same ones (idempotent), each before its own P.V: 4 rows per lane
          uint8_t* vt = sV + stage * Cfg::kTile + one_chunk * kChunkBytes;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int row = lane * 4 + i;
            *reinterpret_cast<uint16_t*>(vt + row * 128 + ((((one_ch >> 3) ^ (row & 7)) << 4) | ((one_ch & 7) << 1))) = one_bits;
          }
          fence_proxy_async_smem();
          __syncwarp();
        }
        mbar_wait(&p_full[x], j & 1);
        tc_fence_after();
        const uint32_t v_addr = smem_u32(sV + stage * Cfg::kTile);
        if (elect_one()) {
#pragma unroll
          for (int ks = 0; ks < BKV / 16; ++ks) {
            const uint32_t pa = pa0 + (ks >> 2) * kChunkBytes + (ks & 3) * 32;
            umma_ss(tO, make_smem_desc_sw128(pa, 16, 1024), make_smem_desc_sw128(v_addr + ks * 2048, kChunkBytes, 1024),
                    idesc_pv, (j | ks) != 0 ? 1u : 0u);
          }
          tc_commit(&v_empty[stage]);
          tc_commit(&o_done[x]);
        }
        __syncwarp();
      }
    }
  } else {
    // ===================== softmax: 4 groups of 4 warps =====================
    const int g = (warp - 4) >> 2;
    const int x = g >> 1;   // query tile A / B
    const int hf = g & 1;   // key half of every tile
    const int ew = warp & 3;
    const int r = ew * 32 + lane;
    const uint32_t lane_off = static_cast<uint32_t>(ew * 32) << 16;
    const uint32_t tS = tmem_base + x * 128 + hf * 64 + lane_off;
    const uint32_t tO = tmem_base + 256 + x * 128 + lane_off;
    uint8_t* prow = sP + x * 2 * kChunkBytes + hf * kChunkBytes + r * 128;
    const int sw = r & 7;
    const float sc = a.scale_log2;
    const int pair_bar = 1 + x * 4 + ew;  // named barrier of the two warps that share these 32 rows
    float m_ref = 0.f;
    for (int j = 0; j < T; ++j) {
      const bool bank = j >= a.n_self_tiles;
      const int len = bank ? a.lb : a.lq;
      const int row0 = (bank ? j - a.n_self_tiles : j) * BKV;
      int valid = len - row0 - hf * 64;  // valid keys in this thread's half
      if (valid > 64) valid = 64;
      mbar_wait(&s_full[x], j & 1);
      tc_fence_after();
      uint32_t sv[2][32];
      tmem_ld_x32(tS, sv[0]);
      tmem_ld_x32(tS + 32, sv[1]);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&s_free[x]);
      // ---- maximum of this half (4 chains), then of the row ----
      float mx0 = -INFINITY, mx1 = -INFINITY, mx2 = -INFINITY, mx3 = -INFINITY;
      if (valid == 64) {
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          mx0 = fmaxf(mx0, __uint_as_float(sv[0][i]));
          mx1 = fmaxf(mx1, __uint_as_float(sv[0][16 + i]));
          mx2 = fmaxf(mx2, __uint_as_float(sv[1][i]));
          mx3 = fmaxf(mx3, __uint_as_float(sv[1][16 + i]));
        }
      } else {
#pragma unroll
        for (int i = 0; i < 64; ++i) {
          if (i >= valid) sv[i >> 5][i & 31] = __float_as_uint(-INFINITY);  // exp2 -> 0: padded keys leave P and the sum
          mx0 = fmaxf(mx0, __uint_as_float(sv[i >> 5][i & 31]));
        }
      }
      float mx = fmaxf(fmaxf(mx0, mx1), fmaxf(mx2, mx3));
      float* mslot = sMax + (((j & 1) * 2 + x) * 2) * 128;
      mslot[hf * 128 + r] = mx;
      asm volatile("bar.sync %0, 64;" ::"r"(pair_bar) : "memory");
      mx = fmaxf(mx, mslot[(hf ^ 1) * 128 + r]) * sc;
      // ---- lazy rescale decision (identical in both halves of a row) ----
      float alpha = 1.0f;
      bool rescale = false;
      if (j == 0) {
        m_ref = mx;
      } else {
        const bool need = mx > m_ref + kRescaleThreshold2;
        rescale = __any_sync(0xffffffffu, need);
        if (need) {
          alpha = ex2f(m_ref - mx);
          m_ref = mx;
        }
      }
      if (j == 0 && x == 1) mbar_wait(stagger, 0);
      // P_X (and O_X) may only be overwritten once the previous P_X.V has retired
      if (j > 0) {
        mbar_wait(&o_done[x], (j - 1) & 1);
        tc_fence_after();
      }
      // ---- probabilities: 16 at a time straight into the swizzled A-operand row ----
      const float nm = -m_ref;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        uint32_t pk[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float p0 = ex2f(fmaf(__uint_as_float(sv[c >> 1][(c & 1) * 16 + 2 * i]), sc, nm));
          const float p1 = ex2f(fmaf(__uint_as_float(sv[c >> 1][(c & 1) * 16 + 2 * i + 1]), sc, nm));
          pk[i] = C::pack(p0, p1);
        }
        *reinterpret_cast<uint4*>(prow + (((2 * c) ^ sw) << 4)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        *reinterpret_cast<uint4*>(prow + (((2 * c + 1) ^ sw) << 4)) = make_uint4(pk[4], pk[5], pk[6], pk[7]);
      }
      if (j == 0 && x == 0) {
        __syncwarp();
        if (lane == 0) mbar_arrive(stagger);
      }
      // ---- correction of O (rare): the two halves split the O columns ----
      if (rescale) {
        const int nc = dpv / 16;
        const int c0 = hf == 0 ? 0 : nc / 2, c1 = hf == 0 ? nc / 2 : nc;
        for (int c = c0; c < c1; ++c) {
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
    // ---- epilogue: O[:, :d] / O[:, d] -> global; the halves split the channel chunks ----
    mbar_wait(&o_done[x], (T - 1) & 1);
    tc_fence_after();
    const int nc = dpv / 16;
    float inv_l;
    {
      uint32_t v[16];
      tmem_ld_x16(tO + (a.d >> 4) * 16, v);
      tmem_ld_wait();
      float l = 0.f;
#pragma unroll
      for (int i = 0; i < 16; ++i)
        if (i == (a.d & 15)) l = __uint_as_float(v[i]);
      inv_l = 1.0f / l;
    }
    const int qrow = q_pair * 2 * BQ + x * BQ + r;
    typename C::T* orow =
        static_cast<typename C::T*>(a.out) + (static_cast<long long>(n) * a.lq + qrow) * a.ld_out + h * a.d;
    const int c0 = hf == 0 ? 0 : (nc + 1) / 2, c1 = hf == 0 ? (nc + 1) / 2 : nc;
    for (int c = c0; c < c1; ++c) {
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
static int launch_pp2(const CUtensorMap& q, const CUtensorMap& k, const CUtensorMap& v, const CUtensorMap& bk,
                      const CUtensorMap& bv, const AttnArgs& a, int n, cudaStream_t st) {
  using Cfg = PP2Cfg<NCH>;
  auto kern = attn_spatial_pp2_kernel<NCH, kBf16>;
  static bool attr_done = false;
  if (!attr_done) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmem);
    if (e != cudaSuccess) return set_cuda_error("cudaFuncSetAttribute(attn_pp2)", e);
    attr_done = true;
  }
  dim3 grid((a.lq + 2 * BQ - 1) / (2 * BQ), a.heads, n);
  cudaError_t e = launch_k(kern, grid, dim3(kPP2Threads), Cfg::kSmem, st, q, k, v, bk, bv, a);
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) return set_cuda_error("attn_pp2 launch", e);
  return MIMO_OK;
}

// the value channels plus the ones column fit one 64-channel chunk: d + 1 <= 64
int launch_attn_pp2(bool bf16, const CUtensorMap& q, const CUtensorMap& k, const CUtensorMap& v, const CUtensorMap& bk,
                    const CUtensorMap& bv, const AttnArgs& a, int n, cudaStream_t st) {
  return bf16 ? launch_pp2<1, true>(q, k, v, bk, bv, a, n, st) : launch_pp2<1, false>(q, k, v, bk, bv, a, n, st);
}

}  // namespace mimo
