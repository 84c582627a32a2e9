"""Tensor-level wrappers over the C ABI. PyTorch is only the owner of device memory and of the stream here:
every function enqueues exactly the kernels of one C entry point on torch's current CUDA stream.

Activations are channels-last 2-D views: [rows, C] with rows = (frame-sample, y, x).

Optional profiling (bench.py): when PROFILE is a list, every call is bracketed by CUDA events on the launching
stream and appends (name, flops, bytes, ev_start, ev_stop) with the call's ALGORITHMIC flops / bytes.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional

import torch

from . import lib as L

_launches = 0  # number of kernels launched through the C ABI (bench.py's gpu_launches)
PROFILE: Optional[List[tuple]] = None


def launches() -> int:
    return _launches


def add_launches(k: int) -> None:
    """Account for kernels launched by a CUDA-graph replay (the graph was recorded from these same wrappers)."""
    global _launches
    _launches += k


class _Call:
    """Counts kernel launches and, when profiling, brackets the call with events."""

    __slots__ = ("name", "k", "flops", "bytes", "e0")

    def __init__(self, name: str, kernels: int = 1, flops: float = 0.0, bytes_: float = 0.0):
        self.name, self.k, self.flops, self.bytes = name, kernels, flops, bytes_

    def __enter__(self):
        global _launches
        _launches += self.k
        if PROFILE is not None:
            self.e0 = torch.cuda.Event(enable_timing=True)
            self.e0.record()
        return self

    def __exit__(self, *exc):
        if PROFILE is not None:
            e1 = torch.cuda.Event(enable_timing=True)
            e1.record()
            PROFILE.append((self.name, self.flops, self.bytes, self.e0, e1))
        return False


def _stream() -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _dt(t: torch.Tensor) -> int:
    if t.dtype == torch.float16:
        return L.F16
    if t.dtype == torch.bfloat16:
        return L.BF16
    raise L.MimoError(f"unsupported dtype {t.dtype}: engine tensors are fp16 or bf16")


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    if t is None:
        return None
    if not t.is_cuda:
        raise L.MimoError("mimo_b200 ops need CUDA tensors (there is no CPU fallback)")
    return t.data_ptr()


def _epilogue(bias=None, rowvec=None, rows_per_group=1, residual=None, scale=1.0, act=L.ACT_NONE) -> L.Epilogue:
    ep = L.Epilogue()
    ep.bias = _ptr(bias)
    ep.rowvec = _ptr(rowvec)
    ep.rows_per_group = int(rows_per_group)
    ep.ld_rowvec = rowvec.stride(0) if rowvec is not None else 0
    ep.residual = _ptr(residual)
    ep.ld_res = residual.stride(0) if residual is not None else 0
    ep.scale = float(scale)
    ep.act = int(act)
    return ep


def gemm(a: torch.Tensor, w: torch.Tensor, out: Optional[torch.Tensor] = None, *, a1: Optional[torch.Tensor] = None,
         bias=None, rowvec=None, rows_per_group=1, residual=None, scale=1.0, act=L.ACT_NONE) -> torch.Tensor:
    """out[M, N(or N/2 for GEGLU)] = epilogue([a | a1][M, K + K1] @ w[N, K + K1]^T)."""
    K1 = a1.shape[1] if a1 is not None else 0
    assert a.dim() == 2 and w.dim() == 2 and a.shape[1] + K1 == w.shape[1]
    assert a.stride(1) == 1 and w.stride(1) == 1
    M, K = a.shape
    N = w.shape[0]
    n_out = N // 2 if act == L.ACT_GEGLU else N
    if out is None:
        out = torch.empty((M, n_out), dtype=a.dtype, device=a.device)
    assert out.shape == (M, n_out) and out.stride(1) == 1
    p = L.GemmParams()
    p.a, p.lda = _ptr(a), a.stride(0)
    p.a1, p.lda1, p.K1 = (_ptr(a1), a1.stride(0), K1) if a1 is not None else (None, 0, 0)
    p.w, p.ldw = _ptr(w), w.stride(0)
    p.out, p.ldo = _ptr(out), out.stride(0)
    p.M, p.N, p.K = M, N, K
    p.dtype = _dt(a)
    p.ep = _epilogue(bias, rowvec, rows_per_group, residual, scale, act)
    kt = K + K1
    with _Call("gemm", 1, 2.0 * M * N * kt, 2.0 * (M * kt + N * kt + M * n_out + (M * N if residual is not None else 0))):
        L.check(L.load().mimo_gemm(C.byref(p), _stream()), "mimo_gemm")
    return out


def conv3x3(x0: torch.Tensor, w: torch.Tensor, n: int, h: int, wd: int, out: Optional[torch.Tensor] = None, *,
            x1: Optional[torch.Tensor] = None, bias=None, rowvec=None, rows_per_group: Optional[int] = None,
            residual=None, scale=1.0, act=L.ACT_NONE) -> torch.Tensor:
    """3x3/s1/p1 conv over channels-last x0 [n*h*wd, c0] (+ x1 [n*h*wd, c1]); w packed [cout, 9*(c0+c1)]."""
    c0 = x0.shape[1]
    c1 = x1.shape[1] if x1 is not None else 0
    cout = w.shape[0]
    assert x0.is_contiguous() and (x1 is None or x1.is_contiguous()) and w.is_contiguous()
    assert w.shape[1] == 9 * (c0 + c1) and x0.shape[0] == n * h * wd
    if out is None:
        out = torch.empty((n * h * wd, cout), dtype=x0.dtype, device=x0.device)
    p = L.Conv3x3Params()
    p.x0, p.c0 = _ptr(x0), c0
    p.x1, p.c1 = _ptr(x1), c1
    p.w = _ptr(w)
    p.out, p.ldo = _ptr(out), out.stride(0)
    p.n, p.h, p.w_, p.cout = n, h, wd, cout
    p.dtype = _dt(x0)
    p.ep = _epilogue(bias, rowvec, rows_per_group or h * wd, residual, scale, act)
    M, cin = n * h * wd, c0 + c1
    with _Call("conv3x3", 1, 2.0 * M * cout * 9 * cin,
               2.0 * (M * cin + 9 * cin * cout + M * cout + (M * cout if residual is not None else 0))):
        L.check(L.load().mimo_conv3x3(C.byref(p), _stream()), "mimo_conv3x3")
    return out


def conv_up2x(x: torch.Tensor, w4: torch.Tensor, n: int, h: int, wd: int, *, bias=None, scale=1.0, act=L.ACT_NONE,
              out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """nearest-x2 upsample + 3x3 conv of channels-last x [n*h*wd, c] -> [n*2h*2wd, cout]; w4 from pack_conv_up2x_weight."""
    c = x.shape[1]
    cout = w4.shape[1]
    assert x.is_contiguous() and w4.is_contiguous() and w4.shape == (4, cout, 4 * c) and x.shape[0] == n * h * wd
    if out is None:
        out = torch.empty((n * 4 * h * wd, cout), dtype=x.dtype, device=x.device)
    p = L.Conv3x3Params()
    p.x0, p.c0 = _ptr(x), c
    p.x1, p.c1 = None, 0
    p.w = _ptr(w4)
    p.out, p.ldo = _ptr(out), out.stride(0)
    p.n, p.h, p.w_, p.cout = n, h, wd, cout
    p.dtype = _dt(x)
    p.ep = _epilogue(bias, None, 1, None, scale, act)
    M = n * h * wd
    # algorithmic work of the REFERENCE op (9 taps on the 4x image); the kernel executes 4/9 of it
    with _Call("conv3x3", 4, 2.0 * 4 * M * cout * 9 * c, 2.0 * (M * c + 16 * c * cout + 4 * M * cout)):
        L.check(L.load().mimo_conv_up2x(C.byref(p), _stream()), "mimo_conv_up2x")
    return out


def im2col3x3(x: torch.Tensor, n: int, h: int, wd: int, *, stride=1, upshift=0, pad_lo=1,
              out: Optional[torch.Tensor] = None) -> torch.Tensor:
    c = x.shape[1]
    uh, uw = h << upshift, wd << upshift
    oh = (uh + 2 * pad_lo - 3 + (0 if pad_lo else 1)) // stride + 1
    ow = (uw + 2 * pad_lo - 3 + (0 if pad_lo else 1)) // stride + 1
    if out is None:
        out = torch.empty((n * oh * ow, 9 * c), dtype=x.dtype, device=x.device)
    with _Call("im2col", 1, 0.0, 2.0 * (x.numel() + out.numel())):
        L.check(L.load().mimo_im2col3x3(_ptr(x), _ptr(out), n, h, wd, c, stride, upshift, pad_lo, out.stride(0),
                                        _dt(x), _stream()), "mimo_im2col3x3")
    return out


def groupnorm(x0: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, n: int, hw: int, *, groups=32,
              eps=1e-5, silu=False, x1: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None,
              stats: Optional[torch.Tensor] = None) -> torch.Tensor:
    c0 = x0.shape[1]
    c1 = x1.shape[1] if x1 is not None else 0
    if out is None:
        out = torch.empty((n * hw, c0 + c1), dtype=x0.dtype, device=x0.device)
    p = L.GroupNormParams()
    p.x0, p.c0 = _ptr(x0), c0
    p.x1, p.c1 = _ptr(x1), c1
    p.gamma, p.beta = _ptr(gamma), _ptr(beta)
    p.out = _ptr(out)
    p.n, p.hw, p.groups = n, hw, groups
    p.eps = float(eps)
    p.silu = int(bool(silu))
    p.dtype = _dt(x0)
    need = L.load().mimo_groupnorm_workspace_bytes(C.byref(p))
    if need < 0:
        L.check(int(need), "mimo_groupnorm_workspace_bytes")
    if stats is None:
        stats = torch.empty(((need + 3) // 4,), dtype=torch.float32, device=x0.device)
    assert x0.is_contiguous() and out.is_contiguous() and stats.numel() * 4 >= need
    p.stats = _ptr(stats)
    with _Call("groupnorm", 2, 0.0, 2.0 * 2 * out.numel()):  # algorithmic: one read + one write
        L.check(L.load().mimo_groupnorm(C.byref(p), _stream()), "mimo_groupnorm")
    return out


def layernorm(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, *, eps=1e-5, pe: Optional[torch.Tensor] = None,
              rows_per_frame=1, frames=1, pe_frame_offset=0, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    assert x.is_contiguous() and x.dim() == 2
    if out is None:
        out = torch.empty_like(x)
    with _Call("layernorm", 1, 0.0, 2.0 * 2 * x.numel()):
        L.check(L.load().mimo_layernorm(_ptr(x), _ptr(gamma), _ptr(beta), _ptr(out), x.shape[0], x.shape[1], float(eps),
                                        _ptr(pe), int(rows_per_frame), int(frames), int(pe_frame_offset), _dt(x),
                                        _stream()), "mimo_layernorm")
    return out


def attn_spatial(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, n: int, lq: int, heads: int, *,
                 bank_k: Optional[torch.Tensor] = None, bank_v: Optional[torch.Tensor] = None,
                 bank_index: Optional[torch.Tensor] = None, scale: Optional[float] = None,
                 out: Optional[torch.Tensor] = None, n_bank_frames: Optional[int] = None) -> torch.Tensor:
    """q/k/v: [n*lq, C] column slices (views) of one fused buffer; bank_k/v: [nb, lb, C]; bank_index int32 [n].
    n_bank_frames (profiling only): how many of the n frames attend to the bank."""
    Cdim = q.shape[1]
    d = Cdim // heads
    assert q.stride(0) == k.stride(0) == v.stride(0) and q.stride(1) == 1
    if out is None:
        out = torch.empty((n * lq, Cdim), dtype=q.dtype, device=q.device)
    p = L.AttnParams()
    p.q, p.k, p.v, p.ld_qkv = _ptr(q), _ptr(k), _ptr(v), q.stride(0)
    lb = 0
    if bank_k is not None:
        assert bank_v is not None and bank_index is not None and bank_index.dtype == torch.int32
        assert bank_k.stride(0) == bank_v.stride(0)
        nb = 1 if bank_k.dim() == 2 else bank_k.shape[0]
        p.bank_k, p.bank_v, p.ld_bank = _ptr(bank_k), _ptr(bank_v), bank_k.stride(-2)
        lb = bank_k.shape[-2]
        p.lb = lb
        p.nb = nb
        p.bank_index = _ptr(bank_index)
    else:
        p.bank_k = p.bank_v = p.bank_index = None
        p.ld_bank, p.lb, p.nb = 0, 0, 0
    p.out, p.ld_out = _ptr(out), out.stride(0)
    p.n, p.lq, p.heads, p.d = n, lq, heads, d
    p.scale = float(scale if scale is not None else d ** -0.5)
    p.dtype = _dt(q)
    nbf = (n if n_bank_frames is None else n_bank_frames) if lb else 0
    with _Call("attn_spatial", 1, 4.0 * Cdim * lq * (n * lq + nbf * lb), 2.0 * (4 * n * lq * Cdim + 2 * lb * Cdim)):
        L.check(L.load().mimo_attn_spatial(C.byref(p), _stream()), "mimo_attn_spatial")
    return out


def attn_temporal(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, batch: int, frames: int, hw: int, heads: int, *,
                  scale: Optional[float] = None, out: Optional[torch.Tensor] = None, q_frames: Optional[int] = None,
                  frames_per_chunk: Optional[int] = None, chunk_stride_rows: int = 0) -> torch.Tensor:
    """q: [batch*q_frames*hw, C]; k/v: column slices of one buffer holding all `frames` frames, possibly as
    frames/frames_per_chunk chunks chunk_stride_rows apart (frame-sharded clip, see the header)."""
    Cdim = q.shape[1]
    d = Cdim // heads
    fq = frames if q_frames is None else q_frames
    if out is None:
        out = torch.empty((batch * fq * hw, Cdim), dtype=q.dtype, device=q.device)
    p = L.AttnTemporalParams()
    p.q, p.ld_q = _ptr(q), q.stride(0)
    p.k, p.v, p.ld_kv = _ptr(k), _ptr(v), k.stride(0)
    assert k.stride(0) == v.stride(0)
    p.out, p.ld_out = _ptr(out), out.stride(0)
    p.chunk_stride_rows = int(chunk_stride_rows)
    p.batch, p.q_frames, p.kv_frames = batch, fq, frames
    p.frames_per_chunk = frames if frames_per_chunk is None else frames_per_chunk
    p.hw, p.heads, p.d = hw, heads, d
    p.scale = float(scale if scale is not None else d ** -0.5)
    p.dtype = _dt(q)
    rows = batch * fq * hw
    with _Call("attn_temporal", 1, 4.0 * rows * frames * Cdim, 2.0 * (2 * rows + 2 * batch * frames * hw) * Cdim):
        L.check(L.load().mimo_attn_temporal(C.byref(p), _stream()), "mimo_attn_temporal")
    return out


def exchange(xg, mode: int, name: str, dst: torch.Tensor, b: int, fl: int, hw: int, Cdim: int,
             residual: Optional[torch.Tensor] = None) -> torch.Tensor:
    """One mimo_exchange of frame group `xg` (host/shard.py: Exchange): pull from every member's source buffer `name`
    into the local tensor `dst` (mode 0 frames->pixels, 1 pixels->frames (+ residual), 2 all-gather)."""
    assert dst.is_contiguous() and (residual is None or (residual.is_contiguous() and residual.shape == dst.shape))
    p = L.ExchangeParams()
    src, flags = xg.bufs[name], xg.flags
    for s in range(xg.G):
        p.peer_src[s] = src.peer_ptrs[s]
        p.peer_ready[s] = flags.peer_ptrs[s]
    p.ctl, p.dst, p.residual = _ptr(xg.ctl), _ptr(dst), _ptr(residual)
    p.mode, p.G, p.r = int(mode), xg.G, xg.r
    p.b, p.fl, p.hw, p.C = int(b), int(fl), int(hw), int(Cdim)
    p.dtype = _dt(dst)
    p.max_blocks, p.timeout_ms = int(xg.max_blocks), int(xg.timeout_ms)
    rows = b * fl * hw * (xg.G if mode == 2 else 1)
    need = b * fl * hw * Cdim * dst.element_size()  # every member's source holds b*fl*hw rows in all three modes
    if need > src.nbytes or dst.numel() != rows * Cdim:
        raise L.MimoError(f"exchange: source buffer '{name}' ({src.nbytes} B) or dst ({tuple(dst.shape)}) does not fit "
                          f"b={b} fl={fl} hw={hw} C={Cdim} mode={mode}")
    with _Call("exchange", 1, 0.0, 2.0 * dst.numel() * dst.element_size() + (dst.numel() * dst.element_size() if residual is not None else 0)):
        L.check(L.load().mimo_exchange(C.byref(p), _stream()), "mimo_exchange")
    return dst


def ncfhw_to_nhwc(src: torch.Tensor, cpad: int, dtype: torch.dtype, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    b, c, f, h, w = src.shape
    assert src.is_contiguous() and src.dtype in (torch.float32, dtype)
    if out is None:
        out = torch.empty((b * f * h * w, cpad), dtype=dtype, device=src.device)
    with _Call("layout", 1, 0.0, src.numel() * src.element_size() + 2.0 * out.numel()):
        L.check(L.load().mimo_ncfhw_to_nhwc(_ptr(src), _ptr(out), b, c, f, h, w, cpad,
                                            int(src.dtype == torch.float32), _dt(out), _stream()), "mimo_ncfhw_to_nhwc")
    return out


def nhwc_to_ncfhw(src: torch.Tensor, b: int, c: int, f: int, h: int, w: int, *, out_dtype: Optional[torch.dtype] = None,
                  out: Optional[torch.Tensor] = None) -> torch.Tensor:
    out_dtype = out_dtype or src.dtype
    if out is None:
        out = torch.empty((b, c, f, h, w), dtype=out_dtype, device=src.device)
    with _Call("layout", 1, 0.0, 2.0 * b * c * f * h * w + out.numel() * out.element_size()):
        L.check(L.load().mimo_nhwc_to_ncfhw(_ptr(src), _ptr(out), b, c, f, h, w, src.stride(0),
                                            int(out.dtype == torch.float32), _dt(src), _stream()), "mimo_nhwc_to_ncfhw")
    return out


def upsample2x(x: torch.Tensor, n: int, h: int, w: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    c = x.shape[1]
    assert x.is_contiguous()
    if out is None:
        out = torch.empty((n * 4 * h * w, c), dtype=x.dtype, device=x.device)
    with _Call("upsample2x", 1, 0.0, 2.0 * 5 * x.numel()):
        L.check(L.load().mimo_upsample2x(_ptr(x), _ptr(out), n, h, w, c, _dt(x), _stream()), "mimo_upsample2x")
    return out


def softmax_rows_(x: torch.Tensor) -> torch.Tensor:
    assert x.dim() == 2 and x.stride(1) == 1
    with _Call("softmax_rows", 1, 0.0, 2.0 * 2 * x.numel()):
        L.check(L.load().mimo_softmax_rows(_ptr(x), x.shape[0], x.shape[1], x.stride(0), _dt(x), _stream()),
                "mimo_softmax_rows")
    return x


def add(a: torch.Tensor, b: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    if out is None:
        out = torch.empty_like(a)
    with _Call("elementwise", 1, 0.0, 2.0 * 3 * a.numel()):
        L.check(L.load().mimo_add(_ptr(a), _ptr(b), _ptr(out), a.numel(), _dt(a), _stream()), "mimo_add")
    return out


def silu(x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    if out is None:
        out = torch.empty_like(x)
    with _Call("elementwise", 1, 0.0, 2.0 * 2 * x.numel()):
        L.check(L.load().mimo_silu(_ptr(x), _ptr(out), x.numel(), _dt(x), _stream()), "mimo_silu")
    return out


def quick_gelu(x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    if out is None:
        out = torch.empty_like(x)
    with _Call("elementwise", 1, 0.0, 2.0 * 2 * x.numel()):
        L.check(L.load().mimo_quick_gelu(_ptr(x), _ptr(out), x.numel(), _dt(x), _stream()), "mimo_quick_gelu")
    return out


def composite_frame(canvas: torch.Tensor, bk: torch.Tensor, mask: torch.Tensor, *, occ: Optional[torch.Tensor] = None,
                    vid: Optional[torch.Tensor] = None, prev: Optional[torch.Tensor] = None, factor: float = 0.0,
                    out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """run_edit.py:282-300 for one frame; uint8 [H, W, 3] images, float32 [H, W] mask, uint8 [H, W] occlusion."""
    for t in (canvas, bk) + tuple(x for x in (occ, vid, prev) if x is not None):
        assert t.dtype == torch.uint8 and t.is_contiguous() and t.is_cuda
    assert mask.dtype == torch.float32 and mask.is_contiguous() and mask.shape == canvas.shape[:2]
    if out is None:
        out = torch.empty_like(canvas)
    px = canvas.shape[0] * canvas.shape[1]
    with _Call("composite", 1, 0.0, float(px * (3 * (3 + (occ is not None) + (prev is not None)) + 4 + (occ is not None)))):
        L.check(L.load().mimo_composite_frame(_ptr(canvas), _ptr(bk), _ptr(mask), _ptr(occ), _ptr(vid), _ptr(prev),
                                              float(factor), _ptr(out), px, _stream()), "mimo_composite_frame")
    return out


def cfg_ddim_step(pred_uncond: torch.Tensor, pred_cond: torch.Tensor, latents: torch.Tensor, guidance: float,
                  sqrt_a_t: float, sqrt_1ma_t: float, sqrt_a_prev: float, sqrt_1ma_prev: float, *,
                  counter: Optional[torch.Tensor] = None, frame_stride: int = 0) -> torch.Tensor:
    """In-place DDIM update of `latents` from the two CFG halves of the (window-accumulated) prediction."""
    assert pred_uncond.is_contiguous() and pred_cond.is_contiguous() and latents.is_contiguous()
    with _Call("cfg_ddim", 1, 0.0, 2.0 * 4 * latents.numel()):
        L.check(L.load().mimo_cfg_ddim_step(_ptr(pred_uncond), _ptr(pred_cond), _ptr(counter), int(frame_stride),
                                            _ptr(latents), latents.numel(), float(guidance), float(sqrt_a_t),
                                            float(sqrt_1ma_t), float(sqrt_a_prev), float(sqrt_1ma_prev), _dt(latents),
                                            _stream()), "mimo_cfg_ddim_step")
    return latents


# ------------------------------------------------------------------------------------------------
# weight packing (host side, once per model load)
# ------------------------------------------------------------------------------------------------
def pack_conv3x3_weight(w: torch.Tensor, cin_pad: Optional[int] = None, cout_pad: Optional[int] = None) -> torch.Tensor:
    """OIHW [cout, cin, 3, 3] -> [cout_pad, 9 * cin_pad], K index = (ky*3+kx) * cin_pad + ch."""
    cout, cin = w.shape[:2]
    cin_pad = cin_pad or (cin + 7) // 8 * 8
    cout_pad = cout_pad or (cout + 7) // 8 * 8
    p = torch.zeros((cout_pad, 9, cin_pad), dtype=w.dtype, device=w.device)
    p[:cout, :, :cin] = w.permute(0, 2, 3, 1).reshape(cout, 9, cin)
    return p.reshape(cout_pad, 9 * cin_pad).contiguous()


def pack_conv_up2x_weight(w: torch.Tensor, b: Optional[torch.Tensor] = None) -> torch.Tensor:
    """OIHW [cout, cin, 3, 3] of the conv that FOLLOWS a nearest-x2 upsampling -> [4, cout_pad, 4 * cin_pad] for
    mimo_conv_up2x: class 2a+b holds, for tap (iy, ix), the sum (in fp32, rounded once) of the 3x3 taps (ky, kx) that read
    source pixel (y - 1 + a + iy, x - 1 + b + ix) when producing output pixel (2y + a, 2x + b)."""
    cout, cin = w.shape[:2]
    cin_pad, cout_pad = (cin + 7) // 8 * 8, (cout + 7) // 8 * 8
    sets = {0: ([0], [1, 2]), 1: ([0, 1], [2])}  # parity -> (taps landing on the first / second source row)
    wf = w.float()
    out = torch.zeros((4, cout_pad, 4, cin_pad), dtype=torch.float32, device=w.device)
    for a in range(2):
        for bb in range(2):
            for iy in range(2):
                for ix in range(2):
                    acc = sum(wf[:, :, ky, kx] for ky in sets[a][iy] for kx in sets[bb][ix])
                    out[2 * a + bb, :cout, 2 * iy + ix, :cin] = acc
    return out.reshape(4, cout_pad, 4 * cin_pad).to(w.dtype).contiguous()


def pack_geglu_weight(w: torch.Tensor, b: Optional[torch.Tensor]):
    """diffusers GEGLU proj weight [2*inner, dim] (value rows then gate rows) -> tile-interleaved rows."""
    n2 = w.shape[0]
    inner = n2 // 2
    g = L.load().mimo_gemm_geglu_granule(n2)
    assert inner % g == 0
    wv, wg = w[:inner].reshape(inner // g, g, -1), w[inner:].reshape(inner // g, g, -1)
    wp = torch.stack([wv, wg], dim=1).reshape(n2, -1).contiguous()
    bp = None
    if b is not None:
        bv, bg = b[:inner].reshape(inner // g, g), b[inner:].reshape(inner // g, g)
        bp = torch.stack([bv, bg], dim=1).reshape(n2).contiguous()
    return wp, bp
