// Spatial self-attention with the reference-image bank: flash attention on tcgen05. This file holds the entry point,
// which picks the kernel by head dim (see attn_common.h), and the single-tile kernel used for d > 128 (the UNet's
// 16x16 and 8x8 levels: d = 160).
//
// One CTA = 128 query rows of one (frame-sample n, head h). The key/value sequence is [self tokens | bank
// tokens of branch bank_index[n]] (bank skipped when bank_index[n] < 0: the unconditional CFG half attends to
// itself only, which is what src/models/mutual_self_attention.py:177-197 computes by running attn1 a second
// time). Per 128-key tile:
//     S  = Q K^T         tcgen05.mma 128x128x(d rounded to 16), Q and K tiles K-major, fp32 S in TMEM
//     P  = exp2(S*c - m) softmax warps: one thread per query row (TMEM lane), online max / sum in fp32,
//                        P written to shared memory as the 128B-swizzled K-major A operand
//     O += P V           tcgen05.mma 128x(d rounded to 16)x128, V tile used as an MN-major B operand
// Q/K/V tiles arrive by 4-D TMA boxes straight out of the fused QKV activation buffer ([token, 3C] rows, head
// slices addressed by a tensor-map dimension); head dims 40/80/160 are zero-filled up to 64-element chunks by
// TMA's out-of-bounds handling, so no padded copies exist in HBM.
// Roles: warp 0 lane 0 TMA, warp 1 lane 0 MMA, warp 2 TMEM alloc, warps 4-7 softmax/correction/epilogue.
#include <cuda_runtime.h>

#include "../../include/mimo_b200.h"
#include "attn_common.h"
#include "host_util.h"
#include "ptx.cuh"

namespace mimo {

constexpr int kAttnThreads = 256;

template <int NCH, int KVST>
struct AttnCfg {
  static constexpr int kQBytes = NCH * kChunkBytes;
  static constexpr int kKVStageBytes = 2 * NCH * kChunkBytes;  // K chunks then V chunks
  static constexpr int kPBytes = 2 * kChunkBytes;
  static constexpr int kSmemBytes = kQBytes + KVST * kKVStageBytes + kPBytes + 1024 + 256;
  static constexpr int kTmemCols = (NCH <= 2) ? 256 : 512;
};

template <int NCH, int KVST, bool kBf16>
__global__ void __launch_bounds__(kAttnThreads)
attn_spatial_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                    const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmBK,
                    const __grid_constant__ CUtensorMap tmBV, AttnArgs a) {
  using Cfg = AttnCfg<NCH, KVST>;
  using C = Cvt<kBf16>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem;
  uint8_t* sKV = sQ + Cfg::kQBytes;
  uint8_t* sP = sKV + KVST * Cfg::kKVStageBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sP + Cfg::kPBytes);
  uint64_t* q_full = bars;
  uint64_t* kv_full = bars + 1;
  uint64_t* kv_empty = kv_full + KVST;
  uint64_t* s_full = kv_empty + KVST;
  uint64_t* p_full = s_full + 1;
  uint64_t* o_done = p_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_done + 1);

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);  // provably warp-uniform for the compiler
  const int lane = threadIdx.x & 31;
  const int q_tile = blockIdx.x;
  const int h = blockIdx.y;
  const int n = blockIdx.z;
  pdl_launch_dependents();
  pdl_wait();
  const int bidx = __shfl_sync(0xffffffffu, a.bank_index ? a.bank_index[n] : -1, 0);
  const int T = a.n_self_tiles + (bidx >= 0 ? a.n_bank_tiles : 0);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmV);
    if (bidx >= 0) {
      tma_prefetch_desc(&tmBK);
      tma_prefetch_desc(&tmBV);
    }
  }
  if (warp == 1 && lane == 0) {
    mbar_init(q_full, 1);
    for (int s = 0; s < KVST; ++s) {
      mbar_init(&kv_full[s], 1);
      mbar_init(&kv_empty[s], 1);
    }
    mbar_init(s_full, 1);
    mbar_init(p_full, 128);
    mbar_init(o_done, 1);
    fence_mbar_init();
  }
  if (warp == 2) tmem_alloc(tmem_slot, Cfg::kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);
  const uint32_t tmem_S = tmem_base;        // 128 fp32 columns
  const uint32_t tmem_O = tmem_base + 128;  // dp fp32 columns

  if (warp == 0 && lane == 0) {
    // ===================== TMA producer =====================
    mbar_expect_tx(q_full, Cfg::kQBytes);
#pragma unroll
    for (int ch = 0; ch < NCH; ++ch) tma_load_4d(sQ + ch * kChunkBytes, &tmQ, q_full, ch * 64, h, q_tile * BQ, n);
    for (int j = 0; j < T; ++j) {
      const int stage = j % KVST;
      const uint32_t phase = (j / KVST) & 1u;
      mbar_wait(&kv_empty[stage], phase ^ 1u);
      uint8_t* sk = sKV + stage * Cfg::kKVStageBytes;
      uint8_t* sv = sk + NCH * kChunkBytes;
      mbar_expect_tx(&kv_full[stage], Cfg::kKVStageBytes);
      const bool bank = j >= a.n_self_tiles;
      const int row0 = (bank ? j - a.n_self_tiles : j) * BKV;
      const int img = bank ? bidx : n;
      const CUtensorMap* mk = bank ? &tmBK : &tmK;
      const CUtensorMap* mv = bank ? &tmBV : &tmV;
#pragma unroll
      for (int ch = 0; ch < NCH; ++ch) {
        tma_load_4d(sk + ch * kChunkBytes, mk, &kv_full[stage], ch * 64, h, row0, img);
        tma_load_4d(sv + ch * kChunkBytes, mv, &kv_full[stage], ch * 64, h, row0, img);
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (whole warp, one elected lane issues: descriptors stay uniform) =====================
    const uint32_t idesc_qk = make_idesc_f16(BQ, BKV, kBf16, false, false);
    const uint32_t idesc_pv = make_idesc_f16(BQ, a.dp, kBf16, false, true);  // B (= V) is MN-major
    const int ksteps_qk = a.dp / 16;
    const uint32_t q_addr = smem_u32(sQ);
    const uint32_t p_addr = smem_u32(sP);
    auto issue_qk = [&](int j) {
      const int stage = j % KVST;
      const uint32_t k_addr = smem_u32(sKV + stage * Cfg::kKVStageBytes);
      if (elect_one()) {
        for (int ks = 0; ks < ksteps_qk; ++ks) {
          const uint32_t off = (ks >> 2) * kChunkBytes + (ks & 3) * 32;
          umma_ss(tmem_S, make_smem_desc_sw128(q_addr + off, 16, 1024), make_smem_desc_sw128(k_addr + off, 16, 1024),
                  idesc_qk, ks != 0 ? 1u : 0u);
        }
        tc_commit(s_full);
      }
      __syncwarp();
    };
    mbar_wait(q_full, 0);
    mbar_wait(&kv_full[0], 0);
    tc_fence_after();
    issue_qk(0);
    for (int j = 0; j < T; ++j) {
      const int stage = j % KVST;
      mbar_wait(p_full, j & 1);
      tc_fence_after();
      const uint32_t v_addr = smem_u32(sKV + stage * Cfg::kKVStageBytes + NCH * kChunkBytes);
      if (elect_one()) {
#pragma unroll
        for (int ks = 0; ks < BKV / 16; ++ks) {
          // A = P: K-major, 64-key chunks of [128 rows x 128 B]; B = V: MN-major, 16 keys = 2 KiB further down
          const uint32_t pa = p_addr + (ks >> 2) * kChunkBytes + (ks & 3) * 32;
          const uint32_t vb = v_addr + ks * 2048;
          umma_ss(tmem_O, make_smem_desc_sw128(pa, 16, 1024), make_smem_desc_sw128(vb, kChunkBytes, 1024), idesc_pv,
                  (j | ks) != 0 ? 1u : 0u);
        }
        tc_commit(&kv_empty[stage]);
        tc_commit(o_done);
      }
      __syncwarp();
      if (j + 1 < T) {
        const int ns = (j + 1) % KVST;
        mbar_wait(&kv_full[ns], ((j + 1) / KVST) & 1u);
        tc_fence_after();
        issue_qk(j + 1);
      }
    }
  } else if (warp >= 4) {
    // ===================== softmax / correction / epilogue =====================
    const int ew = warp & 3;
    const int r = ew * 32 + lane;  // query row inside the tile == TMEM lane
    const uint32_t lane_off = static_cast<uint32_t>(ew * 32) << 16;
    float m = -INFINITY, l = 0.f;
    uint8_t* prow = sP + r * 128;
    const int sw = r & 7;
    for (int j = 0; j < T; ++j) {
      const bool bank = j >= a.n_self_tiles;
      const int len = bank ? a.lb : a.lq;
      const int row0 = (bank ? j - a.n_self_tiles : j) * BKV;
      int valid = len - row0;
      if (valid > BKV) valid = BKV;
      mbar_wait(s_full, j & 1);
      tc_fence_after();
      // pass 1: row maximum
      float mx = -INFINITY;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        uint32_t v[32];
        tmem_ld_x32(tmem_S + lane_off + c * 32, v);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; ++i)
          if (c * 32 + i < valid) mx = fmaxf(mx, __uint_as_float(v[i]));
      }
      const float m_new = fmaxf(m, mx * a.scale_log2);
      const float alpha = exp2f(m - m_new);
      // P (and O) may only be overwritten once the previous P.V has retired
      if (j > 0) {
        mbar_wait(o_done, (j - 1) & 1);
        tc_fence_after();
      }
      // pass 2: probabilities -> swizzled smem (A operand of P.V)
      float rowsum = 0.f;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        uint32_t v[32];
        tmem_ld_x32(tmem_S + lane_off + c * 32, v);
        tmem_ld_wait();
        uint32_t pk[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const int c0 = c * 32 + 2 * i;
          float p0 = 0.f, p1 = 0.f;
          if (c0 < valid) p0 = exp2f(fmaf(__uint_as_float(v[2 * i]), a.scale_log2, -m_new));
          if (c0 + 1 < valid) p1 = exp2f(fmaf(__uint_as_float(v[2 * i + 1]), a.scale_log2, -m_new));
          rowsum += p0 + p1;
          pk[i] = C::pack(p0, p1);
        }
        // 32 keys = 64 B = four 16-byte pieces of this row's 128-B line in chunk (c >> 1)
        uint8_t* line = prow + (c >> 1) * kChunkBytes;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int piece = (c & 1) * 4 + q;
          *reinterpret_cast<uint4*>(line + ((piece ^ sw) << 4)) =
              make_uint4(pk[4 * q], pk[4 * q + 1], pk[4 * q + 2], pk[4 * q + 3]);
        }
      }
      l = l * alpha + rowsum;
      m = m_new;
      // correction: O *= alpha
      if (j > 0) {
        for (int c = 0; c < a.dp / 16; ++c) {
          uint32_t v[16];
          tmem_ld_x16(tmem_O + lane_off + c * 16, v);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = __float_as_uint(__uint_as_float(v[i]) * alpha);
          tmem_st_x16(tmem_O + lane_off + c * 16, v);
        }
        tmem_st_wait();
      }
      fence_proxy_async_smem();
      tc_fence_before();
      mbar_arrive(p_full);
    }
    // epilogue: O / l -> global
    mbar_wait(o_done, (T - 1) & 1);
    tc_fence_after();
    const float inv_l = 1.0f / l;
    const int qrow = q_tile * BQ + r;
    typename C::T* orow =
        static_cast<typename C::T*>(a.out) + (static_cast<long long>(n) * a.lq + qrow) * a.ld_out + h * a.d;
    for (int c = 0; c < a.dp / 16; ++c) {
      uint32_t v[16];
      tmem_ld_x16(tmem_O + lane_off + c * 16, v);
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
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

template <int NCH, int KVST, bool kBf16>
static int launch_attn(const CUtensorMap& q, const CUtensorMap& k, const CUtensorMap& v, const CUtensorMap& bk,
                       const CUtensorMap& bv, const AttnArgs& a, int n, cudaStream_t st) {
  using Cfg = AttnCfg<NCH, KVST>;
  auto kern = attn_spatial_kernel<NCH, KVST, kBf16>;
  static bool attr_done = false;
  if (!attr_done) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes);
    if (e != cudaSuccess) return set_cuda_error("cudaFuncSetAttribute(attn)", e);
    attr_done = true;
  }
  dim3 grid((a.lq + BQ - 1) / BQ, a.heads, n);
  cudaError_t e = launch_k(kern, grid, dim3(kAttnThreads), Cfg::kSmemBytes, st, q, k, v, bk, bv, a);
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) return set_cuda_error("attn launch", e);
  return MIMO_OK;
}

static int attn_tmap(CUtensorMap* m, int dtype, const void* base, int d, int heads, int len, int nimg,
                     long long ld) {
  const uint64_t dims[4] = {static_cast<uint64_t>(d), static_cast<uint64_t>(heads), static_cast<uint64_t>(len),
                            static_cast<uint64_t>(nimg)};
  const uint64_t str[3] = {static_cast<uint64_t>(d) * 2, static_cast<uint64_t>(ld) * 2,
                           static_cast<uint64_t>(len) * ld * 2};
  const uint32_t box[4] = {64, 1, 128, 1};
  return encode_tmap(m, dtype, 4, base, dims, str, box);
}

}  // namespace mimo

using namespace mimo;

extern "C" int mimo_attn_spatial(const mimo_attn_params* p, void* stream) {
  if (!p || !p->q || !p->k || !p->v || !p->out) return set_error(MIMO_ERR_ARG, "mimo_attn_spatial: null pointer");
  if (p->n <= 0 || p->lq <= 0 || p->heads <= 0 || p->d <= 0 || (p->d % 8) || p->d > 192 || (p->ld_qkv % 8) ||
      (p->ld_out % 8))
    return set_error(MIMO_ERR_ARG, "mimo_attn_spatial: need d % 8 == 0, d <= 192, leading dims % 8 == 0");
  const bool has_bank = p->bank_index && p->bank_k && p->bank_v && p->lb > 0;
  if (has_bank && (p->ld_bank % 8)) return set_error(MIMO_ERR_ARG, "mimo_attn_spatial: ld_bank % 8 != 0");
  if (int rc = ensure_device()) return rc;

  AttnArgs a;
  a.lq = p->lq;
  a.lb = has_bank ? p->lb : 0;
  a.heads = p->heads;
  a.d = p->d;
  a.dp = (p->d + 15) / 16 * 16;
  a.n_self_tiles = (p->lq + BKV - 1) / BKV;
  a.n_bank_tiles = has_bank ? (p->lb + BKV - 1) / BKV : 0;
  a.scale_log2 = p->scale * 1.4426950408889634f;
  a.bank_index = has_bank ? p->bank_index : nullptr;
  a.out = p->out;
  a.ld_out = p->ld_out;

  CUtensorMap tq, tk, tv, tbk, tbv;
  if (int rc = attn_tmap(&tq, p->dtype, p->q, p->d, p->heads, p->lq, p->n, p->ld_qkv)) return rc;
  if (int rc = attn_tmap(&tk, p->dtype, p->k, p->d, p->heads, p->lq, p->n, p->ld_qkv)) return rc;
  if (int rc = attn_tmap(&tv, p->dtype, p->v, p->d, p->heads, p->lq, p->n, p->ld_qkv)) return rc;
  if (has_bank) {
    const int nb = p->nb > 0 ? p->nb : 1;
    if (int rc = attn_tmap(&tbk, p->dtype, p->bank_k, p->d, p->heads, p->lb, nb, p->ld_bank)) return rc;
    if (int rc = attn_tmap(&tbv, p->dtype, p->bank_v, p->d, p->heads, p->lb, nb, p->ld_bank)) return rc;
  } else {
    tbk = tk;
    tbv = tv;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const bool bf = p->dtype == MIMO_BF16;
  // d + 1 <= 64 (the 64x64 level, d = 40: MUFU-bound): two softmax threads per row + row sum on the tensor pipe
  // (attn_spatial_pp2.cu; measured 467 vs 429 TFLOP/s)
  if (p->d + 1 <= 64) return launch_attn_pp2(bf, tq, tk, tv, tbk, tbv, a, p->n, st);
  if (a.dp <= 128) return launch_attn_pp(bf, tq, tk, tv, tbk, tbv, a, p->n, st);
  // d <= 192: three 64-wide chunks, one KV stage
  return bf ? launch_attn<3, 1, true>(tq, tk, tv, tbk, tbv, a, p->n, st)
            : launch_attn<3, 1, false>(tq, tk, tv, tbk, tbv, a, p->n, st);
}
