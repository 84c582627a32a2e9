/* mimo_b200 — C ABI of the B200 (sm_100a) denoising-engine kernels.
 *
 * The reference (menyifang/MIMO) has no FFI layer: every op on its hot path is a PyTorch library call made
 * from src/models/*.py. Each entry point below replaces one of those call sites (cited per function as
 * reference file:line) and is what a ctypes binding in the reference's modules would call; see INTEGRATION.md.
 *
 * Conventions
 *  - plain pointers and sizes only; every pointer is a DEVICE pointer unless stated; tensors are dense,
 *    "channels-last": activations are [rows, C] with rows = (frame-sample, y, x) flattened, C contiguous.
 *  - `stream` is a cudaStream_t (CUstream) passed as void*; kernels are enqueued, never synchronised, never
 *    allocate: all entry points are CUDA-graph capturable.
 *  - dtype: 0 = fp16, 1 = bf16 storage; accumulation and all epilogue math are fp32.
 *  - return 0 on success, negative on error; mimo_last_error() gives the thread-local message.
 *  - there is no CPU fallback: on a machine without an sm_100 device every compute entry point fails.
 */
#ifndef MIMO_B200_H_
#define MIMO_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MIMO_OK 0
#define MIMO_ERR_ARG (-1)
#define MIMO_ERR_CUDA (-2)
#define MIMO_ERR_DEVICE (-3)

#define MIMO_F16 0
#define MIMO_BF16 1

#define MIMO_ACT_NONE 0
#define MIMO_ACT_SILU 1
/* GEGLU: weight rows are packed per output tile as [value rows | gate rows]; out has N/2 columns.
 * Packing granule (rows of value, then rows of gate) is returned by mimo_gemm_geglu_granule(). */
#define MIMO_ACT_GEGLU 2

const char* mimo_version(void);
const char* mimo_last_error(void);
/* 0 if device `dev` is sm_100; MIMO_ERR_DEVICE otherwise (also when there is no CUDA device at all). */
int mimo_device_check(int dev);
/* sizeof() of the parameter structs as compiled into the library (0 epilogue, 1 gemm, 2 conv3x3, 3 groupnorm,
 * 4 attn, 5 attn_temporal, 6 exchange): lets a binding verify its struct mirrors before the first call. */
int mimo_abi_sizeof(int which);

/* Fused epilogue shared by GEMM and conv:  out = act((acc + bias[c] + rowvec[row / rows_per_group][c]
 *                                                      + residual[row][c]) * scale)                      */
typedef struct {
  const void* bias;       /* [N] or NULL                                                              */
  const void* rowvec;     /* [ceil(M / rows_per_group), ld_rowvec] or NULL (time embedding / folded cross-attn) */
  int64_t rows_per_group; /* rows sharing one rowvec row (f*H*W for per-CFG-branch vectors)            */
  int64_t ld_rowvec;      /* row stride of rowvec in elements (0 = N)                                  */
  const void* residual;   /* [M, ld_res] or NULL                                                      */
  int64_t ld_res;
  float scale; /* 1 / output_scale_factor                                                  */
  int act;     /* MIMO_ACT_*                                                               */
} mimo_epilogue;

/* out[M,N] = epilogue(A[M,K] . W[N,K]^T).  tcgen05 GEMM, TMA-fed, fp32 accumulate in TMEM.
 * Replaces: torch.nn.Linear / 1x1 Conv2d call sites — to_q/k/v/to_out (diffusers Attention, constructed at
 * src/models/attention.py:321-345, src/models/motion_module.py:282-292), FeedForward/GEGLU
 * (src/models/attention.py:359, motion_module.py:235), proj_in/proj_out (src/models/transformer_3d.py:64-66,
 * 93-95; motion_module.py:122,144), conv_shortcut (src/models/resnet.py:213-215), time_emb_proj (resnet.py:179).
 * Requirements: K % 8 == 0, lda/ldw % 8 == 0, N % 8 == 0, 16-byte aligned bases. */
typedef struct {
  const void* a;
  int64_t lda;
  const void* a1; /* optional second A source: A = [a | a1] along K (virtual concat), or NULL */
  int64_t lda1;
  const void* w;
  int64_t ldw;
  void* out;
  int64_t ldo;
  int32_t M, N, K; /* K = columns of `a`   */
  int32_t K1;      /* columns of `a1` (0 if a1 == NULL); w is [N, K + K1] */
  int32_t dtype;
  mimo_epilogue ep;
} mimo_gemm_params;
int mimo_gemm(const mimo_gemm_params* p, void* stream);
/* number of value rows (== gate rows) per packed GEGLU tile for a packed width N (N = 2 * out features) */
int mimo_gemm_geglu_granule(int32_t N);

/* 3x3 / stride 1 / pad 1 convolution as implicit GEMM: the A operand is fetched tap by tap with 4-D TMA boxes
 * over the NHWC input (out-of-bounds = zero padding), optionally from two tensors (virtual channel concat).
 * Weights packed [Cout, 9 * (c0 + c1)], K index = tap * (c0 + c1) + channel, tap = ky * 3 + kx.
 * Replaces: InflatedConv3d.forward (src/models/resnet.py:9-17) inside ResnetBlock3D (resnet.py:217-247), conv_in /
 * conv_out (src/models/unet_3d_edit_bkfill.py:89-91, 249-251), Upsample3D's conv (resnet.py:88), and the
 * torch.cat([h, skip]) feeding up-block ResBlocks (src/models/unet_3d_blocks.py:697, 827).
 * Requirements: c0 % 8 == 0, c1 % 8 == 0, cout % 8 == 0. */
typedef struct {
  const void* x0;
  int32_t c0;
  const void* x1; /* NULL if single source */
  int32_t c1;
  const void* w;
  void* out;
  int64_t ldo;
  int32_t n, h, w_, cout;
  int32_t dtype;
  mimo_epilogue ep;
} mimo_conv3x3_params;
int mimo_conv3x3(const mimo_conv3x3_params* p, void* stream);
/* Upsample3D (src/models/resnet.py:53-90): nearest x2 (H, W) followed by the 3x3 / pad 1 conv, WITHOUT materialising
 * the upsampled tensor. x0 is the [n, h, w, c0] source, out the [n, 2h, 2w, cout] result (row stride ldo). Output pixel
 * (2y+a, 2x+b) only sees source rows {y-1+a, y+a} and columns {x-1+b, x+b}: four 2x2-tap implicit-GEMM convolutions (one
 * per parity class) whose weights are the sums of the 3x3 taps that land on the same source pixel - 4/9 of the FLOPs.
 * w: [4 classes (2a+b)][cout, 4 * c0], K index = (2*iy + ix) * c0 + channel, packed by the host
 * (mimo_b200.ops.pack_conv_up2x_weight). Epilogue: bias / scale / SiLU only. */
int mimo_conv_up2x(const mimo_conv3x3_params* p, void* stream);

/* im2col gather for the convolutions the TMA path does not cover (stride 2, nearest-x2 upsampled input):
 * col[(n,oy,ox), tap*c + ch] = x[n, (oy*stride-1+ky) >> up, (ox*stride-1+kx) >> up, ch], zero outside.
 * Replaces: Downsample3D (src/models/resnet.py:112-120), F.interpolate in Upsample3D (resnet.py:70-73),
 * PoseGuider's stride-2 convs (src/models/pose_guider.py:31-36). */
int mimo_im2col3x3(const void* x, void* col, int32_t n, int32_t h, int32_t w, int32_t c, int32_t stride,
                   int32_t upshift, int32_t pad_lo, int64_t ldcol, int32_t dtype, void* stream);

/* GroupNorm over channels-last activations, optional SiLU, optional two-source virtual concat. Deterministic: a
 * statistics pass publishes per-slab partial sums, the normalisation pass adds them in a fixed order (no floating-point
 * atomics; bit-identical run to run). stats: workspace of mimo_groupnorm_workspace_bytes(p) bytes, 16-byte aligned,
 * contents irrelevant. Replaces InflatedGroupNorm / nn.GroupNorm + F.silu
 * (src/models/resnet.py:20-28, 220-221, 231, 237; transformer_3d.py:58-60,124; motion_module.py:119-121,156). */
typedef struct {
  const void* x0;
  int32_t c0;
  const void* x1;
  int32_t c1;
  const void* gamma;
  const void* beta; /* [c0 + c1] */
  void* out;        /* [n, hw, c0 + c1] */
  float* stats;
  int32_t n, hw, groups;
  float eps;
  int32_t silu;
  int32_t dtype;
} mimo_groupnorm_params;
int mimo_groupnorm(const mimo_groupnorm_params* p, void* stream);
/* bytes of `stats` workspace mimo_groupnorm needs for these sizes (pointers in *p are ignored); < 0 on bad sizes */
int64_t mimo_groupnorm_workspace_bytes(const mimo_groupnorm_params* p);

/* LayerNorm over the last dim; optional additive per-frame vector AFTER the affine (the motion module's
 * sinusoidal positional encoding): out[r] = LN(x[r]) * gamma + beta + pe[pe_frame_offset + (r / rows_per_frame) % frames]
 * (pe_frame_offset = first global frame of this rank's shard).
 * Replaces nn.LayerNorm (src/models/attention.py:329-360; motion_module.py:230,236) and PositionalEncoding.forward
 * (motion_module.py:277-279). */
int mimo_layernorm(const void* x, const void* gamma, const void* beta, void* out, int64_t rows, int32_t c,
                   float eps, const void* pe, int64_t rows_per_frame, int32_t frames, int32_t pe_frame_offset,
                   int32_t dtype, void* stream);

/* Spatial self-attention with the reference-image bank (flash attention, tcgen05 QK^T and PV, online softmax).
 * q/k/v: [n, lq, heads, d] slices of a fused QKV buffer (row stride ld_qkv elements). bank_k/bank_v:
 * [nb, lb, heads, d] with row stride ld_bank; frame-sample i attends to [self keys | bank keys of branch
 * bank_index[i]] when bank_index[i] >= 0, and to self keys only when bank_index[i] < 0 (the unconditional half).
 * Replaces hacked_basic_transformer_inner_forward's attn1 calls (src/models/mutual_self_attention.py:154-197)
 * -> diffusers Attention/AttnProcessor2_0 -> F.scaled_dot_product_attention. */
typedef struct {
  const void* q;
  const void* k;
  const void* v;
  int64_t ld_qkv;
  const void* bank_k;
  const void* bank_v;
  int64_t ld_bank;
  int32_t lb;                /* bank tokens per feature map */
  int32_t nb;                /* number of bank feature maps (CFG branches written by the reference UNet) */
  const int32_t* bank_index; /* DEVICE [n], values in [-1, nb), or NULL (= no bank) */
  void* out;
  int64_t ld_out;
  int32_t n, lq, heads, d;
  float scale;
  int32_t dtype;
} mimo_attn_params;
int mimo_attn_spatial(const mimo_attn_params* p, void* stream);

/* Temporal self-attention of the motion module: for every (batch b, pixel p, head) a q_frames x kv_frames attention
 * over the frame axis. Query rows are ordered ((b * q_frames + f) * hw + p). Keys/values cover all kv_frames frames
 * and may live in several chunks of frames_per_chunk frames (the per-rank buffers of a frame-sharded clip after the
 * all-gather): kv_row(b, f, p) = (f / frames_per_chunk) * chunk_stride_rows + (b * frames_per_chunk + f %
 * frames_per_chunk) * hw + p. Single GPU: q_frames == kv_frames == frames_per_chunk, chunk_stride_rows = 0.
 * Replaces VersatileAttention.forward (src/models/motion_module.py:353-390), including its two
 * "(b f) d c <-> (b d) f c" transposes. */
typedef struct {
  const void* q;
  int64_t ld_q;
  const void* k;
  const void* v;
  int64_t ld_kv;
  void* out;
  int64_t ld_out;
  int64_t chunk_stride_rows;
  int32_t batch, q_frames, kv_frames, frames_per_chunk;
  int32_t hw, heads, d;
  float scale;
  int32_t dtype;
} mimo_attn_temporal_params;
int mimo_attn_temporal(const mimo_attn_temporal_params* p, void* stream);

/* Frame-shard <-> pixel-shard exchange of the motion module over NVLink PEER MEMORY (one process per GPU, G GPUs in a
 * frame group, this GPU is member r). Each GPU pulls its share directly from its peers' source buffers (IPC-mapped
 * device pointers, see mimo_peer_*), synchronised by epoch flags in peer memory; no collective library and no host
 * work on the data path, CUDA-graph capturable. Tokens are channels-last rows of C elements.
 *   mode 0 (frames -> pixels): src on every peer is [b, fl, hw, C] (its fl frames of the window); dst becomes
 *           [b, G*fl, hw/G, C]: ALL frames of this GPU's pixel shard  (before VersatileAttention, motion_module.py:353-390)
 *   mode 1 (pixels -> frames): src on every peer is [b, G*fl, hw/G, C]; dst becomes [b, fl, hw, C] (+ residual, same
 *           layout as dst): the motion module's output for this GPU's frames (motion_module.py:181-183)
 *   mode 2 (all-gather): src on every peer is [b*fl*hw, C]; dst becomes [G, b*fl*hw, C]
 * peer_src[s] / peer_ready[s]: peer s's source buffer / its array of MIMO_MAX_PEERS uint32 flags (zero-initialised once),
 * as mapped into THIS process; index r is this GPU's own buffer / flags. ctl: two uint32 of local device memory,
 * initialised to {1, 0} once per group, never touched by the host afterwards. All members must issue the same sequence
 * of exchanges. A peer that does not show up within timeout_ms (0 = 30 s) traps the kernel. */
#define MIMO_MAX_PEERS 8
typedef struct {
  const void* peer_src[MIMO_MAX_PEERS];
  void* peer_ready[MIMO_MAX_PEERS];
  void* ctl;
  void* dst;
  const void* residual; /* mode 1 only, or NULL */
  int32_t mode, G, r;
  int32_t b, fl, hw, C;
  int32_t dtype;
  int32_t max_blocks; /* 0 = 2 per SM */
  int32_t timeout_ms;
} mimo_exchange_params;
int mimo_exchange(const mimo_exchange_params* p, void* stream);
/* Peer-shareable device memory for mimo_exchange: cudaMalloc'd, zero-filled, exported as a 64-byte CUDA IPC handle;
 * mimo_peer_open maps another process's buffer into this process for the CURRENT device (peer access is enabled on
 * first use). Bootstrap only (the handles travel over whatever the host uses, e.g. torch.distributed objects). */
int mimo_peer_alloc(int64_t bytes, void** ptr, void* handle64);
int mimo_peer_open(const void* handle64, void** ptr);
int mimo_peer_close(void* ptr);
int mimo_peer_free(void* ptr);

/* Elementwise / layout helpers (each one coalesced pass). */
/* [b, c, f, h, w] (reference layout) -> [(b f), h, w, cpad] channels-last, zero-padding channels c..cpad */
int mimo_ncfhw_to_nhwc(const void* src, void* dst, int32_t b, int32_t c, int32_t f, int32_t h, int32_t w,
                       int32_t cpad, int32_t src_is_f32, int32_t dtype, void* stream);
/* [(b f), h, w, ld] channels-last (first c channels) -> [b, c, f, h, w] */
int mimo_nhwc_to_ncfhw(const void* src, void* dst, int32_t b, int32_t c, int32_t f, int32_t h, int32_t w,
                       int32_t ld, int32_t dst_is_f32, int32_t dtype, void* stream);
/* nearest-neighbour x2 upsampling of [n, h, w, c] -> [n, 2h, 2w, c] (F.interpolate in Upsample3D, resnet.py:70-73) */
int mimo_upsample2x(const void* x, void* out, int32_t n, int32_t h, int32_t w, int32_t c, int32_t dtype, void* stream);
/* in-place row softmax of x[rows, cols] (leading dim ld), fp32 math: the VAE mid-block attention (1 head, d=512) is
 * run as GEMM -> softmax -> GEMM (diffusers AttnProcessor2_0 on UNetMidBlock2D's Attention). */
int mimo_softmax_rows(void* x, int64_t rows, int32_t cols, int64_t ld, int32_t dtype, void* stream);
/* out = a + b (same shape, count elements) */
int mimo_add(const void* a, const void* b, void* out, int64_t count, int32_t dtype, void* stream);
/* out = silu(x) */
int mimo_silu(const void* x, void* out, int64_t count, int32_t dtype, void* stream);

/* out = x * sigmoid(1.702 x): CLIP's quick_gelu (transformers CLIPMLP [3P]; the image encoder of pipeline :378-385) */
int mimo_quick_gelu(const void* x, void* out, int64_t count, int32_t dtype, void* stream);

/* Scene compositing of run_edit.py:282-300, one frame, one pass (all images uint8 [H, W, 3] on the device):
 *   res = canvas * mask + bk * (1 - mask);  [res = res * (1 - occ/255) + vid * (occ/255)];  [out = prev * (1 - factor)
 *   + res * factor];  out -> uint8 by truncation. mask: float32 [H, W] feather mask placed on the full frame; occ: uint8
 *   [H, W] or NULL (then vid is NULL too); prev: the frame composited from the previous, overlapping clip or NULL.
 * Intermediate types follow numpy's promotion in the reference, so the bytes are identical. */
int mimo_composite_frame(const void* canvas, const void* bk, const float* mask, const void* occ, const void* vid,
                         const void* prev, double factor, void* out, int64_t pixels, void* stream);

/* Classifier-free guidance + DDIM (v-prediction, eta = 0) update, one pass:
 *   eps = (pred_u + g * (pred_c - pred_u)) / counter ; x0 = sa_t * x - s1a_t * v ; e = sa_t * v + s1a_t * x ;
 *   x_prev = sa_p * x0 + s1a_p * e.   latents/pred_* are [count]; math in fp32, stored in `dtype`.
 * Replaces pipeline_pose2vid_long_edit_bkfill_roiclip.py:545-553 (+ diffusers DDIMScheduler.step). */
int mimo_cfg_ddim_step(const void* pred_uncond, const void* pred_cond, const void* counter_or_null,
                       int64_t frame_stride, void* latents, int64_t count, float guidance, float sqrt_a_t,
                       float sqrt_1ma_t, float sqrt_a_prev, float sqrt_1ma_prev, int32_t dtype, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MIMO_B200_H_ */
