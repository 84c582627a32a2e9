"""Per-kernel parity on a B200: every C-ABI kernel against a plain PyTorch fp32 reference of the same op, at the
exact shapes of the hot path (SURVEY.md §2.2/§9) and at ragged / tail / empty-ish edge shapes.
Tolerance: rel-L2 <= 2e-3 on fp16 outputs (fp16 rounding of the result is 2^-11 ~ 4.9e-4 relative); integer-valued
GEMM inputs must come out bit-exact."""
import pytest
import torch

pytestmark = pytest.mark.gpu

CHECKS = ["gemm_basic", "gemm_shapes", "gemm_persistent", "gemm_epilogue", "conv_basic", "conv_shapes", "norms",
          "temporal", "elementwise", "spatial_basic", "spatial_shapes"]


@pytest.fixture(scope="module")
def probe():
    if not torch.cuda.is_available():
        pytest.fail("-m gpu tests need a CUDA device: the product path has no CPU fallback")
    from scripts import gpu_probe
    return gpu_probe


@pytest.mark.parametrize("name", CHECKS)
def test_kernel(probe, name):
    assert probe.CHECKS[name](), f"{name} failed (see captured stdout for per-case errors)"
    torch.cuda.synchronize()


def test_two_source_gemm_and_extras(probe):
    from mimo_b200 import ops
    torch.manual_seed(0)
    a0 = torch.randn(300, 1280, device="cuda").half()
    a1 = torch.randn(300, 640, device="cuda").half()
    w = (torch.randn(1280, 1920, device="cuda") / 44).half()
    b = torch.randn(1280, device="cuda").half()
    ref = torch.cat([a0, a1], 1).float() @ w.float().t() + b.float()
    assert probe.report("gemm [a0|a1]", ops.gemm(a0, w, a1=a1, bias=b), ref)
    # odd split (K0 not a multiple of the 64-wide K block): TMA zero fill must keep the two sources apart
    a0, a1 = torch.randn(130, 72, device="cuda").half(), torch.randn(130, 40, device="cuda").half()
    w = torch.randn(64, 112, device="cuda").half() / 10
    assert probe.report("gemm [72|40]", ops.gemm(a0, w, a1=a1), torch.cat([a0, a1], 1).float() @ w.float().t())
    x = torch.randn(2 * 5 * 7, 16, device="cuda").half()
    up = ops.upsample2x(x, 2, 5, 7)
    ref = x.reshape(2, 5, 7, 16).repeat_interleave(2, 1).repeat_interleave(2, 2).reshape(-1, 16)
    assert torch.equal(up, ref)
    s = (torch.randn(37, 4096, device="cuda") * 3).half()
    ref = torch.softmax(s.float(), -1)
    assert probe.report("softmax_rows", ops.softmax_rows_(s.clone()), ref, tol=3e-3)


def test_cfg_ddim_step_matches_torch_fp16_expression():
    """The fused kernel must round where the reference's torch expression rounds (pipeline :545-553)."""
    from mimo_b200 import ops
    from oracle import torch_oracle as O
    torch.manual_seed(1)
    F_, h, w = 5, 8, 8
    lat = torch.randn(1, 4, F_, h, w, device="cuda").half()
    pred = torch.randn(2, 4, F_, h, w, device="cuda").half()
    counter = torch.tensor([1, 2, 1, 2, 2], device="cuda").half()
    d = O.DDIM()
    d.set_timesteps(20)
    for t in (999, 499, 49):
        co = d.coefficients(t)
        got = ops.cfg_ddim_step(pred[0] * counter.view(1, F_, 1, 1), pred[1] * counter.view(1, F_, 1, 1), lat.clone(),
                                3.5, *co, counter=counter, frame_stride=h * w)
        u, c = ((pred * counter.view(1, 1, F_, 1, 1)) / counter.view(1, 1, F_, 1, 1)).chunk(2)
        guided = u + 3.5 * (c - u)
        want = d.step(guided, t, lat)
        assert want.dtype == torch.float16
        diff = (got.float() - want.float()).abs().max()
        assert float(diff) <= 2e-3, (t, float(diff))


def test_conv_up2x_matches_interpolate_plus_conv(probe):
    """Upsample3D (resnet.py:53-90) as four parity-class 2x2-tap convolutions over the source image vs
    F.interpolate(nearest) + conv2d in fp32; UNet and VAE-decoder shapes, ragged widths, SiLU epilogue."""
    import torch.nn.functional as F

    from mimo_b200 import lib as L
    from mimo_b200 import ops
    for n, h, w, cin, cout, act in [(3, 8, 8, 1280, 1280, L.ACT_NONE), (2, 32, 32, 640, 640, L.ACT_NONE),
                                    (1, 64, 64, 512, 512, L.ACT_NONE), (2, 5, 7, 64, 72, L.ACT_SILU),
                                    (1, 130, 3, 16, 8, L.ACT_NONE)]:
        torch.manual_seed(n * 100 + h)
        W = (torch.randn(cout, cin, 3, 3, device="cuda") / (3 * cin ** 0.5)).half()
        b = torch.randn(cout, device="cuda").half()
        x = torch.randn(n, cin, h, w, device="cuda").half()
        ref = F.conv2d(F.interpolate(x.float(), scale_factor=2.0, mode="nearest"), W.float(), b.float(), padding=1)
        if act == L.ACT_SILU:
            ref = F.silu(ref)
        xr = x.permute(0, 2, 3, 1).reshape(n * h * w, cin).contiguous()
        got = ops.conv_up2x(xr, ops.pack_conv_up2x_weight(W), n, h, w, bias=b, act=act)
        got = got.reshape(n, 2 * h, 2 * w, -1)[..., :cout].permute(0, 3, 1, 2)
        assert probe.report(f"conv_up2x n={n} {h}x{w} {cin}->{cout}", got, ref, tol=2e-3)


def test_small_m_long_k(probe):
    """The small-M / long-K problems a frame-sharded GPU sees at the 8x8 and 16x16 levels, with the whole epilogue:
    against fp32 torch and bit-identical run to run."""
    import torch.nn.functional as F

    from mimo_b200 import lib as L
    from mimo_b200 import ops
    torch.manual_seed(5)
    # GEMM with the whole epilogue: bias + per-group row vector + residual + SiLU
    M, N, K = 384, 1280, 5120
    a = (torch.randn(M, K, device="cuda") / 8).half()
    w = (torch.randn(N, K, device="cuda") / 9).half()
    b = torch.randn(N, device="cuda").half()
    rv = torch.randn(2, N, device="cuda").half()
    r = torch.randn(M, N, device="cuda").half()
    ref = F.silu(a.float() @ w.float().t() + b.float() + rv.float().repeat_interleave(192, 0) + r.float())
    got = ops.gemm(a, w, bias=b, rowvec=rv, rows_per_group=192, residual=r, act=L.ACT_SILU)
    got2 = ops.gemm(a, w, bias=b, rowvec=rv, rows_per_group=192, residual=r, act=L.ACT_SILU)
    assert torch.equal(got, got2)
    assert probe.report("gemm 384x1280x5120", got, ref)
    # 3x3 convolution, two sources (up-block concat), time-embedding row vector, residual
    n, h, c0, c1, co = 6, 8, 1280, 1280, 1280
    x0 = torch.randn(n * h * h, c0, device="cuda").half()
    x1 = torch.randn(n * h * h, c1, device="cuda").half()
    Wc = (torch.randn(co, c0 + c1, 3, 3, device="cuda") / (3 * (c0 + c1) ** 0.5)).half()
    bias = torch.randn(co, device="cuda").half()
    tv = torch.randn(2, co, device="cuda").half()
    res = torch.randn(n * h * h, co, device="cuda").half()
    xin = torch.cat([x0, x1], 1).float().reshape(n, h, h, c0 + c1).permute(0, 3, 1, 2)
    ref = F.conv2d(xin, Wc.float(), bias.float(), padding=1).permute(0, 2, 3, 1).reshape(n * h * h, co)
    ref = ref + tv.float().repeat_interleave(3 * h * h, 0) + res.float()
    wp = ops.pack_conv3x3_weight(Wc)
    got = ops.conv3x3(x0, wp, n, h, h, x1=x1, bias=bias, rowvec=tv, rows_per_group=3 * h * h, residual=res)
    got2 = ops.conv3x3(x0, wp, n, h, h, x1=x1, bias=bias, rowvec=tv, rows_per_group=3 * h * h, residual=res)
    assert torch.equal(got, got2)
    assert probe.report("conv 6x8x8 2560->1280", got, ref)
