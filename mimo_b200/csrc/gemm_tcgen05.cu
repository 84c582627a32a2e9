// Persistent, warp-specialised tcgen05 GEMM / implicit-GEMM 3x3 convolution for sm_100a.
//
//   D[M,N] = epilogue( A[M,K] . W[N,K]^T )          fp16/bf16 operands, fp32 accumulate in TMEM
//
// One CTA per SM loops over 128 x BN output tiles (static round-robin schedule, n-tile fastest so that CTAs
// running concurrently share A tiles in L2). Every byte that crosses the SM boundary moves by TMA; no thread issues
// a scattered global load or store on the steady-state path. Roles (512 threads; the producer / issuer warps run
// their loops with all 32 lanes and elect one lane per TMA / tcgen05 instruction, which keeps addresses and
// descriptors in uniform registers):
//   warp 0        : TMA producer   - ring of {A 128x64, W BNx64} 128B-swizzled stages
//   warp 1        : MMA issuer     - tcgen05.mma.cta_group::1.kind::f16 128xBNx16; accumulators double-buffered in
//                                    TMEM so the epilogue of tile i overlaps the main loop of tile i+1
//   warp 2        : TMEM allocator
//   warp 3        : residual producer (kRes) - TMA boxes of the residual tensor, 128 rows x 32 columns each, into a
//                                    private ring of 8 KiB slots per epilogue group
//   warps 4..15   : epilogue       - three groups of 4 warps deal out the tile's 32-column chunks. Per chunk:
//                                    tcgen05.ld 32 lanes x 32 columns -> acc * scale + column constants (bias +
//                                    per-branch vector, staged in smem one tile ahead) + residual (smem ring)
//                                    -> SiLU / GEGLU -> 64B-swizzled staging buffer -> TMA store
// Convolution mode replaces the A loads by 4-D TMA boxes {64 ch, TW, TH, TN} over the NHWC input, one box per
// (tap, 64-channel block, source tensor); TMA's out-of-bounds zero fill is the conv's zero padding and also
// the K tail, and the output / residual boxes use the same {TW, TH, TN} footprint (stores are clipped at image
// borders). Two source tensors give the up-blocks' channel concat without materialising it.
#include <cuda_runtime.h>

#include <type_traits>
#include <cudaTypedefs.h>

#include "../../include/mimo_b200.h"
#include "host_util.h"
#include "ptx.cuh"

namespace mimo {

constexpr int BM = 128;
constexpr int BK = 64;  // 64 x 16-bit = one 128-byte swizzle row
constexpr int kEpiGroups = 3;                        // epilogue warpgroups (4 warps each), splitting a tile's chunks
constexpr int kGemmThreads = 128 + kEpiGroups * 128;  // warps 0-3: TMA / MMA / TMEM / residual; then the epilogue
// chunk range of epilogue group g when n chunks are dealt out as evenly as possible
__host__ __device__ constexpr int grp_count(int n, int g) { return n / kEpiGroups + (g < n % kEpiGroups ? 1 : 0); }
__host__ __device__ constexpr int grp_base(int n, int g) {
  return g * (n / kEpiGroups) + (g < n % kEpiGroups ? g : n % kEpiGroups);
}
constexpr int kChunk = 8192;  // one 128-row x 32-column (64 B) epilogue chunk

struct EpiArgs {
  const void* bias;
  const void* rowvec;
  long long rows_per_group;
  long long ld_rowvec;
  float scale;
  int act;
  long long* trace;  // debug (mimo_debug_gemm_trace): clock64 timeline of CTA 0, or nullptr
};

struct ConvGeom {
  int conv;  // 0: plain GEMM rows; 1: rows are (n, y, x) footprints
  int H, W, NI;
  int TW, TH, TN;
  int tiles_w, tiles_h;
  int ctot;         // c0 + c1
  int c0;           // channels of source 0 (GEMM mode: K of source 0)
  int kb0, kb1;     // 64-wide K blocks (per tap in conv mode) of source 0 / 1
  int a_bytes;      // bytes one A box deposits in shared memory
  int chunk_bytes;  // bytes one output / residual box moves (TW*TH*TN rows x 64 B)
  int ntaps;        // 9 (3x3) or 4 (one parity class of nearest-x2 upsample + 3x3, see mimo_conv_up2x)
  signed char tdx[9], tdy[9];  // input offset of tap t relative to the output pixel
};

template <int BN, bool kRes>
struct GemmCfg {
  static constexpr int kStageBytes = BM * BK * 2 + BN * BK * 2;
  static constexpr int kNChunk = BN / 32;
  static constexpr int kOutBytes = kEpiGroups * 2 * kChunk;  // per epilogue group: double buffer
  static constexpr int kResPerGroup = BN >= 256 ? 1 : 2;  // private ring of each epilogue group
  static constexpr int kResSlots = kRes ? kEpiGroups * kResPerGroup : 0;
  static constexpr int kResBytes = kResSlots * kChunk;
  static constexpr int kBarBytes = 512;
  static constexpr int kFixed = kBarBytes + 2048 /*sbias*/ + kOutBytes + kResBytes;
  static constexpr int kMaxStages = (BN >= 256) ? 4 : (BN >= 160 ? 5 : (BN >= 128 ? 6 : 8));
  static constexpr int kFit = (227 * 1024 - kFixed) / kStageBytes;
  static constexpr int kStages = kFit < kMaxStages ? kFit : kMaxStages;
  static constexpr int kTmemCols = (2 * BN <= 128) ? 128 : (2 * BN <= 256 ? 256 : 512);
  static constexpr int kSmemBytes = kStages * kStageBytes + kFixed;
  static_assert(kStages >= 3, "pipeline too shallow");
};

template <int BN, bool kBf16, bool kRes>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_tcgen05_kernel(const __grid_constant__ CUtensorMap tmA0, const __grid_constant__ CUtensorMap tmA1,
                    const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmOut,
                    const __grid_constant__ CUtensorMap tmRes, int M, int N, int num_m_tiles, int num_n_tiles,
                    int num_k_blocks, ConvGeom g, EpiArgs ep) {
  using Cfg = GemmCfg<BN, kRes>;
  using C = Cvt<kBf16>;
  using T = typename C::T;
  constexpr int NCHUNK = Cfg::kNChunk;
  extern __shared__ __align__(1024) uint8_t smem[];  // 128B-swizzled tiles need 1024-byte alignment
  uint8_t* sOut = smem + Cfg::kStages * Cfg::kStageBytes;  // [2 groups][2 buffers][8 KiB]
  uint8_t* sRes = sOut + Cfg::kOutBytes;                    // [kResSlots][8 KiB]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sRes + Cfg::kResBytes);
  uint64_t* full_bar = bars;         // kStages (<= 8)
  uint64_t* empty_bar = bars + 8;    // kStages
  uint64_t* tmem_full = bars + 16;   // 2
  uint64_t* tmem_empty = bars + 18;  // 2
  uint64_t* res_full = bars + 20;    // kResSlots (<= 8)
  uint64_t* res_empty = bars + 28;   // kResSlots
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 36);
  float* sbias = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(bars) + Cfg::kBarBytes);  // [2][256]

  pdl_launch_dependents();
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);  // provably warp-uniform for the compiler
  const int lane = threadIdx.x & 31;
  const int num_tiles = num_m_tiles * num_n_tiles;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA0);
    tma_prefetch_desc(&tmA1);
    tma_prefetch_desc(&tmB);
    tma_prefetch_desc(&tmOut);
    if (kRes) tma_prefetch_desc(&tmRes);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < Cfg::kStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tmem_full[b], 1);
      mbar_init(&tmem_empty[b], kEpiGroups * 4);
    }
    for (int s = 0; s < Cfg::kResSlots; ++s) {
      mbar_init(&res_full[s], 1);
      mbar_init(&res_empty[s], 4);
    }
    fence_mbar_init();
  }
  if (warp == 2) tmem_alloc(tmem_slot, Cfg::kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);
  pdl_wait();  // everything above touched only shared memory / TMEM / the kernel parameters

  // tile -> coordinates of its first output row / pixel
  auto tile_origin = [&](int m_tile, int& x0, int& y0, int& n0) {
    if (g.conv) {
      x0 = (m_tile % g.tiles_w) * g.TW;
      y0 = ((m_tile / g.tiles_w) % g.tiles_h) * g.TH;
      n0 = (m_tile / (g.tiles_w * g.tiles_h)) * g.TN;
    } else {
      x0 = y0 = n0 = 0;
    }
  };

  // Producer and issuer warps run their loops with all 32 lanes (uniform control flow) and elect one lane for the
  // TMA / tcgen05 instructions: addresses and descriptors then live in uniform registers. A lane-0-only branch makes
  // the compiler treat them as divergent and wrap every instruction in a ~20-instruction election loop - ~150 clk per
  // MMA, more than a 128x256x16 MMA takes.
  if (warp == 0) {
    // ===================== TMA producer (operands) =====================
    // (all index arithmetic is incremental: this warp has ~300 clk per k-block and runs at ~5 clk per instruction
    // next to the epilogue warps of its sub-partition - divisions here used to throttle the 3x3 convolutions)
    uint32_t it = 0, stage = 0, phase = 0;
    const int kb_per_tap = g.kb0 + g.kb1;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      const int m_tile = tile / num_n_tiles;
      const int n_tile = tile % num_n_tiles;
      int x0, y0, n0;
      tile_origin(m_tile, x0, y0, n0);
      // conv: k-block inside the tap, tap index / offsets, tap * ctot
      int tap = 0, rem = 0;
      int dx = g.tdx[0], dy = g.tdy[0], tap_k = 0;
      for (int kb = 0; kb < num_k_blocks; ++kb, ++it) {
        mbar_wait(&empty_bar[stage], phase ^ 1u);
        if (ep.trace && blockIdx.x == 0 && lane == 0 && it < 512) ep.trace[2560 + it] = clock64();
        uint8_t* sa = smem + stage * Cfg::kStageBytes;
        uint8_t* sb = sa + BM * BK * 2;
        if (elect_one()) {
          if (!g.conv) {
            mbar_expect_tx(&full_bar[stage], BM * BK * 2 + BN * BK * 2);
            if (kb < g.kb0) {  // A = [A0 | A1] along K (virtual concat for the up-block shortcut GEMMs)
              tma_load_2d(sa, &tmA0, &full_bar[stage], kb * BK, m_tile * BM);
              tma_load_2d(sb, &tmB, &full_bar[stage], kb * BK, n_tile * BN);
            } else {
              tma_load_2d(sa, &tmA1, &full_bar[stage], (kb - g.kb0) * BK, m_tile * BM);
              tma_load_2d(sb, &tmB, &full_bar[stage], g.c0 + (kb - g.kb0) * BK, n_tile * BN);
            }
          } else {
            mbar_expect_tx(&full_bar[stage], g.a_bytes + BN * BK * 2);
            int kcoord;
            if (rem < g.kb0) {
              tma_load_4d(sa, &tmA0, &full_bar[stage], rem * BK, x0 + dx, y0 + dy, n0);
              kcoord = tap_k + rem * BK;
            } else {
              tma_load_4d(sa, &tmA1, &full_bar[stage], (rem - g.kb0) * BK, x0 + dx, y0 + dy, n0);
              kcoord = tap_k + g.c0 + (rem - g.kb0) * BK;
            }
            tma_load_2d(sb, &tmB, &full_bar[stage], kcoord, n_tile * BN);
          }
        }
        __syncwarp();
        if (++rem == kb_per_tap) {
          rem = 0;
          tap_k += g.ctot;
          if (++tap == g.ntaps) tap = 0;
          dx = g.tdx[tap];
          dy = g.tdy[tap];
        }
        if (++stage == Cfg::kStages) {
          stage = 0;
          phase ^= 1u;
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    constexpr uint32_t idesc = make_idesc_f16(BM, BN, kBf16, false, false);
    uint32_t lt = 0, stage = 0, phase = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++lt) {
      const uint32_t acc = lt & 1u;
      const uint32_t acc_phase = (lt >> 1) & 1u;
      mbar_wait(&tmem_empty[acc], acc_phase ^ 1u);
      tc_fence_after();
      long long* trm = (ep.trace && blockIdx.x == 0 && lane == 0 && lt < 32) ? ep.trace + 2048 + lt * 16 : nullptr;
      if (trm) trm[0] = clock64();
      const uint32_t d_tmem = tmem_base + acc * BN;
      for (int kb = 0; kb < num_k_blocks; ++kb) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        if (trm && kb < 12) trm[1 + kb] = clock64();
        const uint32_t sa = smem_u32(smem + stage * Cfg::kStageBytes);
        const uint32_t sb = sa + BM * BK * 2;
        const uint64_t da = make_smem_desc_sw128(sa, 16, 1024);
        const uint64_t db = make_smem_desc_sw128(sb, 16, 1024);
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            // advance 16 elements (32 B) along K inside the 128-B swizzle row: +2 in the (addr >> 4) field
            umma_ss(d_tmem, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
          }
          tc_commit(&empty_bar[stage]);  // frees the smem stage once these MMAs have read it
          if (kb == num_k_blocks - 1) tc_commit(&tmem_full[acc]);  // accumulator complete -> epilogue
        }
        __syncwarp();
        if (++stage == Cfg::kStages) {
          stage = 0;
          phase ^= 1u;
        }
      }
      if (trm) trm[14] = clock64();
    }
  } else if (warp == 3) {
    // ===================== TMA producer (residual chunks) =====================
    if constexpr (kRes) {
      // Each epilogue column group owns a private ring of slots (a barrier shared by consumers that can
      // sit in different phases would let the later one alias a completed phase of the same parity).
      constexpr int SH = Cfg::kResPerGroup;
      constexpr int IMAX = grp_count(NCHUNK, 0);
      uint32_t cnt[kEpiGroups] = {};
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int m_tile = tile / num_n_tiles;
        const int n_tile = tile % num_n_tiles;
        int x0, y0, n0;
        tile_origin(m_tile, x0, y0, n0);
        for (int i = 0; i < IMAX; ++i) {
#pragma unroll
          for (int h = 0; h < kEpiGroups; ++h) {
            if (i >= grp_count(NCHUNK, h)) continue;
            const int c = grp_base(NCHUNK, h) + i;
            const uint32_t k = cnt[h]++;
            const uint32_t slot = h * SH + k % SH;
            mbar_wait(&res_empty[slot], ((k / SH) & 1u) ^ 1u);
            if (elect_one()) {
              mbar_expect_tx(&res_full[slot], g.chunk_bytes);
              const int col = n_tile * BN + c * 32;  // boxes beyond N are zero-filled (keeps the slot sequence uniform)
              if (g.conv)
                tma_load_4d(sRes + slot * kChunk, &tmRes, &res_full[slot], col, x0, y0, n0);
              else
                tma_load_2d(sRes + slot * kChunk, &tmRes, &res_full[slot], col, m_tile * BM);
            }
            __syncwarp();
          }
        }
      }
    }
  } else if (warp >= 4) {
    // ===================== epilogue (8 warps) =====================
    // warp w may only touch TMEM lanes [32*(w%4), +32): warps 4-7 and 8-11 each cover all 128 rows; the two groups
    // split the tile's 32-column chunks between them.
    const int ew = warp & 3;
    const int hsel = (warp - 4) >> 2;
    const int r = ew * 32 + lane;
    const bool issuer = (ew == 0) && (lane == 0);
    const int sw = (r >> 1) & 3;  // 64-byte swizzle: 16-byte piece index ^= address bits [7:8]
    uint8_t* obuf_base = sOut + hsel * 2 * kChunk;
    const int bar_id = 2 + hsel;
    const bool do_silu = ep.act == MIMO_ACT_SILU;
    uint32_t lt = 0, oc = 0, rc = 0;
    long long* tr = (ep.trace && blockIdx.x == 0 && ew == 0 && lane == 0) && hsel < 2 ? ep.trace + hsel * 1024 : nullptr;
    int tk = 0;
#define GEMM_TR() do { if (tr && lt < 32 && tk < 32) tr[lt * 32 + tk++] = clock64(); } while (0)
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++lt) {
      tk = 0;
      GEMM_TR();  // 0: tile start
      const int m_tile = tile / num_n_tiles;
      const int n_tile = tile % num_n_tiles;
      const uint32_t acc = lt & 1u;
      const uint32_t acc_phase = (lt >> 1) & 1u;
      int x0, y0, n0;
      tile_origin(m_tile, x0, y0, n0);

      // ---- rows of this tile; which group(s) of the per-branch vector they belong to ----
      // (32-bit arithmetic: M, the pixel count and rows_per_group all fit an int; 64-bit divisions cost ~1 us here)
      const uint32_t rpg = static_cast<uint32_t>(ep.rows_per_group);
      long long row = 0;
      bool row_ok = true;
      if (!g.conv) {
        row = static_cast<long long>(m_tile) * BM + r;
        row_ok = row < M;
      } else {
        const int x = r % g.TW, y = (r / g.TW) % g.TH, n = r / (g.TW * g.TH);
        row_ok = (n < g.TN) && (x0 + x < g.W) && (y0 + y < g.H) && (n0 + n < g.NI);
        row = (static_cast<long long>(n0 + n) * g.H + (y0 + y)) * g.W + (x0 + x);
      }
      // first / last group touched by a tile (uniform per tile)
      auto tile_groups = [&](int mt, uint32_t& gf, uint32_t& gl) {
        if (!g.conv) {
          const uint32_t m0 = static_cast<uint32_t>(mt) * BM;
          uint32_t m1 = m0 + BM - 1;
          if (m1 > static_cast<uint32_t>(M) - 1) m1 = static_cast<uint32_t>(M) - 1;
          gf = m0 / rpg;
          gl = m1 / rpg;
        } else {
          int tx, ty, tn;
          tile_origin(mt, tx, ty, tn);
          int n1 = tn + g.TN - 1;
          if (n1 > g.NI - 1) n1 = g.NI - 1;
          const uint32_t hw = static_cast<uint32_t>(g.H) * g.W;
          gf = (static_cast<uint32_t>(tn) * hw) / rpg;
          gl = (static_cast<uint32_t>(n1 + 1) * hw - 1) / rpg;
        }
      };
      // column constants of a tile: bias (+ the per-branch vector when the whole tile shares one group)
      const int ce = (warp - 4) * 32 + lane;  // one column per epilogue thread (BN <= 256)
      auto load_consts = [&](int t) -> float {
        float v = 0.f;
        const int mt = t / num_n_tiles, nt = t % num_n_tiles;
        const int col = nt * BN + ce;
        if (ce < BN && col < N) {
          if (ep.bias) v = C::to_f(static_cast<const T*>(ep.bias)[col]);
          if (ep.rowvec) {
            uint32_t gf, gl;
            tile_groups(mt, gf, gl);
            if (gf == gl) v += C::to_f(static_cast<const T*>(ep.rowvec)[static_cast<long long>(gf) * ep.ld_rowvec + col]);
          }
        }
        return ep.act == MIMO_ACT_GEGLU ? v : v * ep.scale;  // y = acc * scale + (bias + vec) * scale
      };
      bool rv_uniform = false;
      if (ep.rowvec) {
        uint32_t gf, gl;
        tile_groups(m_tile, gf, gl);
        rv_uniform = gf == gl;
      }
      float* sb = sbias + acc * 256;
      if (lt == 0 && ce < BN) sb[ce] = load_consts(tile);  // later tiles: staged at the end of the previous tile
      asm volatile("bar.sync 1, %0;" ::"n"(kEpiGroups * 128) : "memory");  // epilogue warps only: constants visible, previous tile retired
      GEMM_TR();  // 1: column constants staged
      // constants of the next tile: the loads fly under this tile's chunks
      const int next_tile = tile + gridDim.x;
      float next_const = 0.f;
      if (next_tile < num_tiles) next_const = load_consts(next_tile);
      const T* rv = (ep.rowvec && !rv_uniform && row_ok)
                        ? static_cast<const T*>(ep.rowvec) + static_cast<long long>(static_cast<uint32_t>(row) / rpg) * ep.ld_rowvec
                        : nullptr;
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(ew * 32) << 16) + acc * BN;

      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after();
      GEMM_TR();  // 2: accumulator ready

      if (ep.act != MIMO_ACT_GEGLU) {
        const int cbase = grp_base(NCHUNK, hsel);
        const int ccount = grp_count(NCHUNK, hsel);
        const float scale = ep.scale;
        // one 32-column chunk; the activation is a compile-time tag so the element loop is branch-free
        // kMode 0: no column constants, unit scale, no residual -> accumulators are packed as they are;
        //       1: y = acc * scale + consts (+ residual);  2: as 1, plus per-row vectors (tile straddles groups)
        auto chunk = [&](int c, auto silu_tag, auto mode_tag) {
          constexpr bool kSilu = decltype(silu_tag)::value;
          constexpr int kMode = decltype(mode_tag)::value;
          uint8_t* obuf = obuf_base + (oc & 1u) * kChunk;
          ++oc;
          GEMM_TR();  // chunk +0
          uint32_t v[32];
          tmem_ld_x32(taddr + c * 32, v);
          float4 cb[8];
          if constexpr (kMode != 0) {  // constants land in registers while the TMEM load is in flight
#pragma unroll
            for (int q = 0; q < 8; ++q) cb[q] = *reinterpret_cast<const float4*>(sb + c * 32 + q * 4);
          }
          [[maybe_unused]] const uint8_t* rrow = nullptr;
          [[maybe_unused]] uint32_t rslot = 0;
          if constexpr (kRes) {
            constexpr int SH = Cfg::kResPerGroup;
            const uint32_t k = rc++;
            rslot = hsel * SH + k % SH;
            mbar_wait(&res_full[rslot], (k / SH) & 1u);
            rrow = sRes + rslot * kChunk + r * 64;
          }
          tmem_ld_wait();
          GEMM_TR();  // chunk +1: accumulators (and residual) in registers
          const int col0 = n_tile * BN + c * 32;
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            float f[8];
            if constexpr (kMode == 0) {
#pragma unroll
              for (int j = 0; j < 8; ++j) f[j] = __uint_as_float(v[q * 8 + j]);
            } else {
              const float4 b0 = cb[2 * q], b1 = cb[2 * q + 1];
              float cst[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
              if constexpr (kMode == 2) {
                // the per-row vector joins the column constants FIRST, exactly as load_consts() pre-sums them when a
                // tile lies inside one group: acc + (bias + vec) either way, so a tile that straddles two CFG branches
                // and one that does not round identically (sharded == un-sharded, bit for bit)
                if (rv && col0 + q * 8 < N) {
                  const uint4 b = __ldg(reinterpret_cast<const uint4*>(rv + col0 + q * 8));
                  const uint32_t bw[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
                  for (int j = 0; j < 4; ++j) {
                    const float2 t = C::unpack(bw[j]);
                    cst[2 * j] = fmaf(t.x, scale, cst[2 * j]);
                    cst[2 * j + 1] = fmaf(t.y, scale, cst[2 * j + 1]);
                  }
                }
              }
#pragma unroll
              for (int j = 0; j < 8; ++j) f[j] = fmaf(__uint_as_float(v[q * 8 + j]), scale, cst[j]);
            }
            if constexpr (kRes) {
              const uint4 rr = *reinterpret_cast<const uint4*>(rrow + ((q ^ sw) << 4));
              const uint32_t bw[4] = {rr.x, rr.y, rr.z, rr.w};
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const float2 t = C::unpack(bw[j]);
                f[2 * j] = fmaf(t.x, scale, f[2 * j]);
                f[2 * j + 1] = fmaf(t.y, scale, f[2 * j + 1]);
              }
            }
            if constexpr (kSilu) {
#pragma unroll
              for (int j = 0; j < 8; ++j) f[j] = silu_f(f[j]);
            }
            uint4 o;
            o.x = C::pack(f[0], f[1]);
            o.y = C::pack(f[2], f[3]);
            o.z = C::pack(f[4], f[5]);
            o.w = C::pack(f[6], f[7]);
            *reinterpret_cast<uint4*>(obuf + r * 64 + ((q ^ sw) << 4)) = o;
          }
          if constexpr (kRes) {
            __syncwarp();
            if (lane == 0) mbar_arrive(&res_empty[rslot]);
          }
          GEMM_TR();  // chunk +2: staged
          fence_proxy_async_smem();
          if (issuer) tma_store_wait_read0();  // see "Staging-buffer reuse" below
          GEMM_TR();  // chunk +3: fenced, previous store has left shared memory
          asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");
          GEMM_TR();  // chunk +4: group barrier
          if (issuer) {
            if (g.conv)
              tma_store_4d(&tmOut, obuf, col0, x0, y0, n0);
            else
              tma_store_2d(&tmOut, obuf, col0, m_tile * BM);
            tma_store_commit();
          }
        };
        using M0 = std::integral_constant<int, 0>;
        using M1 = std::integral_constant<int, 1>;
        using M2 = std::integral_constant<int, 2>;
        const bool need_rv = ep.rowvec != nullptr && !rv_uniform;  // uniform per tile
        const bool plain = !kRes && !do_silu && !need_rv && ep.bias == nullptr && ep.rowvec == nullptr && scale == 1.0f;
        // not unrolled: the per-tile code has to stay resident in the instruction cache (fully unrolled, with the
        // activation / row-vector variants, it was ~80 KB and every warp crawled at ~6 clk per instruction)
        if (plain) {
#pragma unroll 1
          for (int i = 0; i < ccount; ++i) chunk(cbase + i, std::false_type{}, M0{});
        } else if (need_rv) {
          if (do_silu) {
#pragma unroll 1
            for (int i = 0; i < ccount; ++i) chunk(cbase + i, std::true_type{}, M2{});
          } else {
#pragma unroll 1
            for (int i = 0; i < ccount; ++i) chunk(cbase + i, std::false_type{}, M2{});
          }
        } else if (do_silu) {
#pragma unroll 1
          for (int i = 0; i < ccount; ++i) chunk(cbase + i, std::true_type{}, M1{});
        } else {
#pragma unroll 1
          for (int i = 0; i < ccount; ++i) chunk(cbase + i, std::false_type{}, M1{});
        }
      } else {
        // GEGLU: tile columns [0, BN/2) are values, [BN/2, BN) the matching gates; 32-column pairs are split
        // dealt out to the epilogue groups.
        constexpr int HALF = BN / 2;
        constexpr int NPAIR = HALF / 32;
        const int pbase = grp_base(NPAIR, hsel);
        const int pcount = grp_count(NPAIR, hsel);
#pragma unroll 1
        for (int i = 0; i < pcount; ++i) {
          {
            const int c = pbase + i;
            uint8_t* obuf = obuf_base + (oc & 1u) * kChunk;
            ++oc;
            uint32_t v[32], gt[32];
            tmem_ld_x32(taddr + c * 32, v);
            tmem_ld_x32(taddr + HALF + c * 32, gt);
            tmem_ld_wait();
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              float f[8];
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                const float fv = __uint_as_float(v[q * 8 + j]) + sb[c * 32 + q * 8 + j];
                const float fg = __uint_as_float(gt[q * 8 + j]) + sb[HALF + c * 32 + q * 8 + j];
                f[j] = fv * gelu_erf_fast(fg);
              }
              uint4 o;
              o.x = C::pack(f[0], f[1]);
              o.y = C::pack(f[2], f[3]);
              o.z = C::pack(f[4], f[5]);
              o.w = C::pack(f[6], f[7]);
              *reinterpret_cast<uint4*>(obuf + r * 64 + ((q ^ sw) << 4)) = o;
            }
            fence_proxy_async_smem();
            if (issuer) tma_store_wait_read0();
            asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");
            if (issuer) {
              tma_store_2d(&tmOut, obuf, n_tile * HALF + c * 32, m_tile * BM);
              tma_store_commit();
            }
          }
        }
      }
      if (next_tile < num_tiles && ce < BN) sbias[(acc ^ 1u) * 256 + ce] = next_const;
      // all TMEM reads of this accumulator buffer are complete (wait::ld above): hand it back to the MMA warp
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[acc]);
    }
    if (issuer) tma_store_wait_all();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

// Staging-buffer reuse: a group's two 8 KiB buffers alternate per chunk. The issuer executes
// cp.async.bulk.wait_group.read 0 just BEFORE it joins barrier(i) - after its own math of chunk i, so the ~700 clk a
// store needs to drain shared memory hide under that math - i.e. after it committed store(i-1); every thread writes
// buffer (i+1)&1 only after barrier(i), by which time stores <= i-1 - including store(i-1), the last reader of that
// buffer - have finished reading shared memory.

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
struct Maps {
  CUtensorMap a0, a1, b, out, res;
};

template <int BN, bool kBf16, bool kRes>
static int launch_cfg(const Maps& m, int M, int N, int mt, int nt, int nkb, const ConvGeom& g, const EpiArgs& ep,
                      cudaStream_t st) {
  using Cfg = GemmCfg<BN, kRes>;
  auto kern = gemm_tcgen05_kernel<BN, kBf16, kRes>;
  static bool attr_done = false;  // per instantiation
  if (!attr_done) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes);
    if (e != cudaSuccess) return set_cuda_error("cudaFuncSetAttribute(gemm)", e);
    attr_done = true;
  }
  const int tiles = mt * nt;
  const int grid = tiles < num_sms() ? tiles : num_sms();
  cudaError_t e = launch_k(kern, dim3(grid), dim3(kGemmThreads), Cfg::kSmemBytes, st, m.a0, m.a1, m.b, m.out, m.res, M, N, mt,
                           nt, nkb, g, ep);
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) return set_cuda_error("gemm launch", e);
  return MIMO_OK;
}

template <bool kBf16>
static int launch_bn(int bn, bool res, const Maps& m, int M, int N, int mt, int nt, int nkb, const ConvGeom& g,
                     const EpiArgs& ep, cudaStream_t st) {
  switch (bn) {
    case 64:
      return res ? launch_cfg<64, kBf16, true>(m, M, N, mt, nt, nkb, g, ep, st)
                 : launch_cfg<64, kBf16, false>(m, M, N, mt, nt, nkb, g, ep, st);
    case 128:
      return res ? launch_cfg<128, kBf16, true>(m, M, N, mt, nt, nkb, g, ep, st)
                 : launch_cfg<128, kBf16, false>(m, M, N, mt, nt, nkb, g, ep, st);
    case 160:
      return res ? launch_cfg<160, kBf16, true>(m, M, N, mt, nt, nkb, g, ep, st)
                 : launch_cfg<160, kBf16, false>(m, M, N, mt, nt, nkb, g, ep, st);
    case 192:
      return res ? launch_cfg<192, kBf16, true>(m, M, N, mt, nt, nkb, g, ep, st)
                 : launch_cfg<192, kBf16, false>(m, M, N, mt, nt, nkb, g, ep, st);
    case 256:
      return res ? launch_cfg<256, kBf16, true>(m, M, N, mt, nt, nkb, g, ep, st)
                 : launch_cfg<256, kBf16, false>(m, M, N, mt, nt, nkb, g, ep, st);
  }
  return set_error(MIMO_ERR_ARG, "gemm: unsupported BN");
}

static int g_force_bn = 0;
static long long* g_gemm_trace = nullptr;  // test hook (mimo_debug_gemm_trace)

// Tile-width choice: least padded columns first, then the widest tile (fewer A re-reads, higher MMA N).
int pick_bn(int N, bool geglu, long long m_tiles) {
  if (g_force_bn) return g_force_bn;
  if (geglu) {
    if (N % 256 == 0) return 256;
    if (N % 128 == 0) return 128;
    return 64;
  }
  const int cands[5] = {256, 192, 160, 128, 64};
  int best = 64;
  double best_eff = -1.0;
  for (int i = 0; i < 5; ++i) {
    const int bn = cands[i];
    const int nt = (N + bn - 1) / bn;
    double eff = static_cast<double>(N) / (static_cast<double>(nt) * bn);
    // small problems: prefer enough tiles to occupy the machine
    const long long tiles = m_tiles * nt;
    if (tiles < num_sms() && bn > 64) eff *= 0.5 + 0.5 * static_cast<double>(tiles) / num_sms();
    if (eff > best_eff + 1e-9) {
      best_eff = eff;
      best = bn;
    }
  }
  return best;
}

static EpiArgs make_epi(const mimo_epilogue& e, int N) {
  EpiArgs a;
  a.bias = e.bias;
  a.rowvec = e.rowvec;
  a.rows_per_group = e.rows_per_group > 0 ? e.rows_per_group : 1;
  if (a.rows_per_group > 0x7fffffffLL) a.rows_per_group = 0x7fffffffLL;  // row counts are ints: same grouping
  a.ld_rowvec = e.ld_rowvec > 0 ? e.ld_rowvec : N;
  a.scale = e.scale;
  a.act = e.act;
  a.trace = g_gemm_trace;
  return a;
}

}  // namespace mimo

using namespace mimo;

extern "C" int mimo_debug_force_bn(int bn) {
  g_force_bn = bn;
  return 0;
}
extern "C" int mimo_debug_gemm_trace(void* buf) {  // >= 4096 int64 of device memory, or NULL
  g_gemm_trace = static_cast<long long*>(buf);
  return 0;
}

extern "C" int mimo_gemm_geglu_granule(int32_t N) { return pick_bn(N, true, 1 << 20) / 2; }

extern "C" int mimo_gemm(const mimo_gemm_params* p, void* stream) {
  if (!p || !p->a || !p->w || !p->out) return set_error(MIMO_ERR_ARG, "mimo_gemm: null pointer");
  if (p->M <= 0 || p->N <= 0 || p->K <= 0) return set_error(MIMO_ERR_ARG, "mimo_gemm: empty problem");
  if ((p->K % 8) || (p->lda % 8) || (p->ldw % 8) || (p->N % 8) || (p->ldo % 8))
    return set_error(MIMO_ERR_ARG, "mimo_gemm: K, N, lda, ldw, ldo must be multiples of 8");
  if (p->ep.residual && (p->ep.ld_res % 8)) return set_error(MIMO_ERR_ARG, "mimo_gemm: ld_res % 8 != 0");
  const bool geglu = p->ep.act == MIMO_ACT_GEGLU;
  if (geglu && (p->ep.residual || p->ep.rowvec))
    return set_error(MIMO_ERR_ARG, "mimo_gemm: GEGLU takes neither a residual nor a row vector");
  if (int rc = ensure_device()) return rc;
  const int mt = (p->M + BM - 1) / BM;
  const int K1 = p->a1 ? p->K1 : 0;
  if (K1 < 0 || (K1 % 8) || (p->a1 && (p->lda1 % 8))) return set_error(MIMO_ERR_ARG, "mimo_gemm: K1/lda1 % 8 != 0");
  const int kb0 = (p->K + BK - 1) / BK;
  const int kb1 = (K1 + BK - 1) / BK;
  const int nkb = kb0 + kb1;
  const int bn = pick_bn(p->N, geglu, mt);
  if (geglu && (p->N % bn)) return set_error(MIMO_ERR_ARG, "mimo_gemm: GEGLU needs N % tile == 0");
  const int nt = (p->N + bn - 1) / bn;
  const bool res = p->ep.residual != nullptr && !geglu;

  Maps m;
  const uint64_t adim[2] = {static_cast<uint64_t>(p->K), static_cast<uint64_t>(p->M)};
  const uint64_t astr[1] = {static_cast<uint64_t>(p->lda) * 2};
  const uint32_t abox[2] = {BK, BM};
  if (int rc = encode_tmap(&m.a0, p->dtype, 2, p->a, adim, astr, abox)) return rc;
  m.a1 = m.a0;
  if (K1) {
    const uint64_t a1dim[2] = {static_cast<uint64_t>(K1), static_cast<uint64_t>(p->M)};
    const uint64_t a1str[1] = {static_cast<uint64_t>(p->lda1) * 2};
    if (int rc = encode_tmap(&m.a1, p->dtype, 2, p->a1, a1dim, a1str, abox)) return rc;
  }
  const uint64_t bdim[2] = {static_cast<uint64_t>(p->K + K1), static_cast<uint64_t>(p->N)};
  const uint64_t bstr[1] = {static_cast<uint64_t>(p->ldw) * 2};
  const uint32_t bbox[2] = {BK, static_cast<uint32_t>(bn)};
  if (int rc = encode_tmap(&m.b, p->dtype, 2, p->w, bdim, bstr, bbox)) return rc;
  // output / residual: 128-row x 32-column boxes, 64-byte swizzle
  const int n_out = geglu ? p->N / 2 : p->N;
  const uint64_t odim[2] = {static_cast<uint64_t>(n_out), static_cast<uint64_t>(p->M)};
  const uint64_t ostr[1] = {static_cast<uint64_t>(p->ldo) * 2};
  const uint32_t obox[2] = {32, BM};
  if (int rc = encode_tmap(&m.out, p->dtype, 2, p->out, odim, ostr, obox, 64)) return rc;
  m.res = m.out;
  if (res) {
    const uint64_t rstr[1] = {static_cast<uint64_t>(p->ep.ld_res) * 2};
    if (int rc = encode_tmap(&m.res, p->dtype, 2, p->ep.residual, odim, rstr, obox, 64)) return rc;
  }

  ConvGeom g = {};
  g.kb0 = kb0;
  g.kb1 = kb1;
  g.c0 = p->K;
  g.chunk_bytes = kChunk;
  const EpiArgs ep = make_epi(p->ep, p->N);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  return p->dtype == MIMO_BF16 ? launch_bn<true>(bn, res, m, p->M, p->N, mt, nt, nkb, g, ep, st)
                               : launch_bn<false>(bn, res, m, p->M, p->N, mt, nt, nkb, g, ep, st);
}

// One implicit-GEMM convolution launch: `ntaps` taps at offsets (tdx, tdy) over the [n, h, w, c] input(s); the output
// (and residual) pixel (n, y, x) lives at out + ((n * oh + y * sy) * ow + x * sx) * ldo elements, i.e. a strided view of a
// larger image when (sx, sy) != (1, 1).
static int conv_launch(const mimo_conv3x3_params* p, const void* w, int ntaps, const signed char* tdx,
                       const signed char* tdy, void* out, int sx, int sy, int ow, int oh, void* stream) {
  const int c1 = p->x1 ? p->c1 : 0;
  ConvGeom g = {};
  g.conv = 1;
  g.H = p->h;
  g.W = p->w_;
  g.NI = p->n;
  g.TW = p->w_ < BM ? p->w_ : BM;
  g.TH = BM / g.TW;
  if (g.TH > p->h) g.TH = p->h;
  if (g.TH < 1) g.TH = 1;
  g.TN = BM / (g.TW * g.TH);
  if (g.TN > p->n) g.TN = p->n;
  if (g.TN < 1) g.TN = 1;
  if (g.TN > 1 && g.TH != p->h) g.TN = 1;  // several images per tile only when a tile spans whole images
  g.tiles_w = (p->w_ + g.TW - 1) / g.TW;
  g.tiles_h = (p->h + g.TH - 1) / g.TH;
  const int tiles_n = (p->n + g.TN - 1) / g.TN;
  g.ctot = p->c0 + c1;
  g.c0 = p->c0;
  g.kb0 = (p->c0 + BK - 1) / BK;
  g.kb1 = (c1 + BK - 1) / BK;
  g.a_bytes = g.TW * g.TH * g.TN * BK * 2;
  g.chunk_bytes = g.TW * g.TH * g.TN * 64;
  g.ntaps = ntaps;
  for (int t = 0; t < 9; ++t) {
    g.tdx[t] = t < ntaps ? tdx[t] : 0;
    g.tdy[t] = t < ntaps ? tdy[t] : 0;
  }
  const int mt = g.tiles_w * g.tiles_h * tiles_n;
  const int nkb = ntaps * (g.kb0 + g.kb1);
  const long long Mrows = static_cast<long long>(p->n) * p->h * p->w_;
  if (Mrows > 0x7fffffffLL) return set_error(MIMO_ERR_ARG, "mimo_conv: too many pixels");
  const int bn = pick_bn(p->cout, false, mt);
  const int nt = (p->cout + bn - 1) / bn;
  const bool res = p->ep.residual != nullptr;

  Maps m;
  auto nhwc_map = [&](CUtensorMap* tm, const void* base, int c, long long pitch, uint32_t box_c, int swz, int px,
                      int py, int iw, int ih) {
    // pixel (n, y, x) at base + ((n * ih + y * py) * iw + x * px) * pitch elements
    const uint64_t dim[4] = {static_cast<uint64_t>(c), static_cast<uint64_t>(p->w_), static_cast<uint64_t>(p->h),
                             static_cast<uint64_t>(p->n)};
    const uint64_t str[3] = {static_cast<uint64_t>(px) * pitch * 2, static_cast<uint64_t>(py) * iw * pitch * 2,
                             static_cast<uint64_t>(ih) * iw * pitch * 2};
    const uint32_t box[4] = {box_c, static_cast<uint32_t>(g.TW), static_cast<uint32_t>(g.TH),
                             static_cast<uint32_t>(g.TN)};
    return encode_tmap(tm, p->dtype, 4, base, dim, str, box, swz);
  };
  if (int rc = nhwc_map(&m.a0, p->x0, p->c0, p->c0, BK, 128, 1, 1, p->w_, p->h)) return rc;
  m.a1 = m.a0;
  if (c1)
    if (int rc = nhwc_map(&m.a1, p->x1, c1, c1, BK, 128, 1, 1, p->w_, p->h)) return rc;
  {
    const uint64_t dim[2] = {static_cast<uint64_t>(ntaps) * g.ctot, static_cast<uint64_t>(p->cout)};
    const uint64_t str[1] = {static_cast<uint64_t>(ntaps) * g.ctot * 2};
    const uint32_t box[2] = {BK, static_cast<uint32_t>(bn)};
    if (int rc = encode_tmap(&m.b, p->dtype, 2, w, dim, str, box)) return rc;
  }
  if (int rc = nhwc_map(&m.out, out, p->cout, p->ldo, 32, 64, sx, sy, ow, oh)) return rc;
  m.res = m.out;
  if (res)
    if (int rc = nhwc_map(&m.res, p->ep.residual, p->cout, p->ep.ld_res, 32, 64, 1, 1, p->w_, p->h)) return rc;

  const EpiArgs ep = make_epi(p->ep, p->cout);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  return p->dtype == MIMO_BF16 ? launch_bn<true>(bn, res, m, static_cast<int>(Mrows), p->cout, mt, nt, nkb, g, ep, st)
                               : launch_bn<false>(bn, res, m, static_cast<int>(Mrows), p->cout, mt, nt, nkb, g, ep, st);
}

static int conv_check(const mimo_conv3x3_params* p, const char* who) {
  if (!p || !p->x0 || !p->w || !p->out) return set_error(MIMO_ERR_ARG, "mimo_conv: null pointer");
  if (p->n <= 0 || p->h <= 0 || p->w_ <= 0 || p->cout <= 0 || p->c0 <= 0)
    return set_error(MIMO_ERR_ARG, "mimo_conv: empty problem");
  const int c1 = p->x1 ? p->c1 : 0;
  if ((p->c0 % 8) || (c1 % 8) || (p->cout % 8) || (p->ldo % 8))
    return set_error(MIMO_ERR_ARG, "mimo_conv: channel counts must be multiples of 8");
  if (p->ep.act == MIMO_ACT_GEGLU) return set_error(MIMO_ERR_ARG, "mimo_conv: GEGLU not supported");
  if (p->ep.residual && (p->ep.ld_res % 8)) return set_error(MIMO_ERR_ARG, "mimo_conv: ld_res % 8 != 0");
  (void)who;
  return ensure_device();
}

extern "C" int mimo_conv3x3(const mimo_conv3x3_params* p, void* stream) {
  if (int rc = conv_check(p, "mimo_conv3x3")) return rc;
  static const signed char dx[9] = {-1, 0, 1, -1, 0, 1, -1, 0, 1};
  static const signed char dy[9] = {-1, -1, -1, 0, 0, 0, 1, 1, 1};
  return conv_launch(p, p->w, 9, dx, dy, p->out, 1, 1, p->w_, p->h, stream);
}

// nearest-x2 upsampling followed by a 3x3 / pad 1 convolution, without the upsampled tensor: output pixel (2y+a, 2x+b)
// only ever sees the 2x2 source neighbourhood {y-1+a, y+a} x {x-1+b, x+b}, so each of the four parity classes (a, b) is a
// 2x2-tap convolution over the SOURCE image whose weights are sums of the 3x3 taps that land on the same source pixel
// (packed by the host: w = [4 classes][cout, 4 * cin], class = 2a + b, tap = 2 iy + ix). 4/9 of the FLOPs, no 4x buffer.
extern "C" int mimo_conv_up2x(const mimo_conv3x3_params* p, void* stream) {
  if (int rc = conv_check(p, "mimo_conv_up2x")) return rc;
  if (p->ep.residual || p->ep.rowvec) return set_error(MIMO_ERR_ARG, "mimo_conv_up2x: bias / activation epilogue only");
  const int ctot = p->c0 + (p->x1 ? p->c1 : 0);
  const size_t esz = 2;
  for (int a = 0; a < 2; ++a)
    for (int b = 0; b < 2; ++b) {
      const signed char dx[4] = {static_cast<signed char>(b - 1), static_cast<signed char>(b),
                                 static_cast<signed char>(b - 1), static_cast<signed char>(b)};
      const signed char dy[4] = {static_cast<signed char>(a - 1), static_cast<signed char>(a - 1),
                                 static_cast<signed char>(a), static_cast<signed char>(a)};
      const char* w = static_cast<const char*>(p->w) + static_cast<size_t>(2 * a + b) * p->cout * 4 * ctot * esz;
      char* out = static_cast<char*>(p->out) + (static_cast<size_t>(a) * 2 * p->w_ + b) * p->ldo * esz;
      if (int rc = conv_launch(p, w, 4, dx, dy, out, 2, 2, 2 * p->w_, 2 * p->h, stream)) return rc;
    }
  return MIMO_OK;
}
