"""BASELINE.json configs[0]: "run_animate.py 1-frame 256x256, 2 DDIM steps, fp32 device=cpu (plumbing, no GPU)".

THIS repo's sampler (mimo_b200/host/pipeline.py: preprocess + sample_tensors — byte-level image path, deduplicated
backgrounds, joint VAE encode, conditional-half reference pass, context windows, fused CFG+DDIM call) executed on the CPU
with the engine entry points replaced, in this test only, by oracle-backed stand-ins (the product has no CPU path), against
the golden clip the reference's own pipeline produced (tests/golden/pipeline_cfg1.pt). Every line of host logic between the
public inputs and the engine calls runs for real; the kernels behind those calls are pinned on the GPU."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle.dropin import oracle_engines  # same stand-ins as the drop-in proof


class _Event:
    def __init__(self, enable_timing=False):
        pass

    def record(self):
        pass

    def elapsed_time(self, other):
        return 0.0


def own_sampler_clip(monkeypatch, golden_dir, F_, guidance):
    """One clip of this repo's sampler over oracle-backed engines: BASELINE configs[0] (F_ = 1) or the 26-frame,
    two-window case at 64x64 (then also the same clip from oracle.sample_clip as `ref_out`)."""
    import PIL.Image
    from transformers import CLIPVisionConfig, CLIPVisionModelWithProjection

    from mimo_b200 import ops
    from mimo_b200.host import modules as M
    from mimo_b200.host.pipeline import Pose2VideoPipeline, pil_to_tensor
    from mimo_b200.host.scheduler import DDIMScheduler
    from oracle import torch_oracle as O
    g = torch.load(golden_dir / "pipeline_cfg1.pt")
    seed, size, steps = g["seed"], g["size"], g["steps"]
    if F_ != 1:
        seed, size = 300, 64  # the 26-frame / two-window case: compared with oracle.sample_clip instead of a fixture
    widths = (128, 256, 512, 512)
    cfg = O.UNetConfig(block_out_channels=widths)
    vcfg = O.VAEConfig(block_out_channels=tuple(g["vae_widths"]) if F_ == 1 else (32, 64, 128, 128))
    oracle_engines(monkeypatch, O, cfg, vcfg)
    monkeypatch.setattr(torch.cuda, "Event", _Event)

    def cfg_ddim(pu, pc, latents, guidance, sa_t, s1a_t, sa_p, s1a_p, *, counter=None, frame_stride=0):
        u, c = pu, pc
        if counter is not None:
            u, c = u / counter.view(1, -1, 1, 1), c / counter.view(1, -1, 1, 1)
        v = u + guidance * (c - u)
        x = latents[0]
        x0 = sa_t * x - s1a_t * v
        eps = sa_t * v + s1a_t * x
        latents[0] = sa_p * x0 + s1a_p * eps
        return latents

    monkeypatch.setattr(ops, "cfg_ddim_step", cfg_ddim)
    mk = dict(num_attention_heads=8, num_transformer_block=1, attention_block_types=["Temporal_Self", "Temporal_Self"],
              temporal_position_encoding=True, temporal_position_encoding_max_len=32, temporal_attention_dim_div=1)
    den = M.UNet3DConditionModel(block_out_channels=widths, cross_attention_dim=768, use_inflated_groupnorm=True,
                                 use_motion_module=True, motion_module_mid_block=True, motion_module_type="Vanilla",
                                 motion_module_kwargs=mk)
    ref = M.UNet2DConditionModel(block_out_channels=widths, cross_attention_dim=768)
    pg = M.PoseGuider(widths[0], 3, (16, 32, 96, 256))
    vae = M.AutoencoderKL(block_out_channels=vcfg.block_out_channels)
    sds = dict(den=O.make_denoising_unet_sd(cfg, seed), ref=O.make_reference_unet_sd(cfg, seed + 1),
               pg=O.make_pose_guider_sd(seed + 2, widths[0]), vae=O.make_vae_sd(vcfg, seed + 3))
    for m, k in ((den, "den"), (ref, "ref"), (pg, "pg"), (vae, "vae")):
        m.load_state_dict(sds[k], strict=True)
    torch.manual_seed(seed + 4)
    clip = CLIPVisionModelWithProjection(CLIPVisionConfig(hidden_size=64, intermediate_size=128, num_hidden_layers=2,
                                                          num_attention_heads=4, image_size=224, patch_size=32,
                                                          projection_dim=cfg.cross_attention_dim)).eval()
    sched = DDIMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", clip_sample=False,
                          steps_offset=1, prediction_type="v_prediction", rescale_betas_zero_snr=True,
                          timestep_spacing="trailing")
    pipe = Pose2VideoPipeline(vae=vae, image_encoder=clip, reference_unet=ref, denoising_unet=den, pose_guider=pg,
                              scheduler=sched)
    monkeypatch.setattr(Pose2VideoPipeline, "_clip", lambda self: type("C", (), {
        "image_embeds": staticmethod(lambda px: clip(px).image_embeds)})())
    # the stand-in denoising engine lacks the two attributes the sampler manages on the real one
    eng = den.engine()
    eng.xchg, eng._graphs = None, {}
    rng = np.random.RandomState(seed)
    ref_img = PIL.Image.fromarray(rng.randint(0, 256, (size, size, 3), dtype=np.uint8))
    poses, bks = [], []
    for i in range(F_):
        a = np.zeros((size, size, 3), np.uint8)
        a[size // 4: size // 2 + i % 8, size // 3: size // 3 + 40] = rng.randint(11, 256, 3)
        poses.append(PIL.Image.fromarray(a))
        bks.append(PIL.Image.fromarray(rng.randint(0, 256, (size, size, 3), dtype=np.uint8)))
    with torch.no_grad():
        host = pipe.preprocess(ref_img, poses, bks, size, size, F_, torch.manual_seed(42), torch.float32)
        seen, never = [], []
        out = pipe.sample_tensors(host, steps, guidance, callback=lambda i, t, lat: seen.append((i, int(t), tuple(lat.shape))))
        pipe.sample_tensors(host, 1, guidance, callback=lambda *a: never.append(a), callback_steps=2, decode=False)
    ref_out = None
    if F_ != 1:
        with torch.no_grad():
            emb = clip(pipe._clip_pixels(ref_img)).image_embeds
            lat0 = torch.randn((1, 4, F_, size // 8, size // 8), generator=torch.manual_seed(42), dtype=torch.float32)
            W = O.Weights(sds["den"], sds["ref"], sds["pg"], sds["vae"], cfg, vcfg)
            ref_out = O.sample_clip(W, pil_to_tensor(ref_img, size, size, True),
                                    pil_to_tensor(poses, size, size, False).permute(1, 0, 2, 3).unsqueeze(0),
                                    pil_to_tensor(bks, size, size, True), emb, lat0, steps, guidance)
    return SimpleNamespace(out=out, seen=seen, never=never, ref_out=ref_out, golden=g, size=size, den=den)


@pytest.mark.parametrize("F_,guidance", [(1, 3.5), (26, 3.5), (26, 1.0)])
def test_own_sampler_host_logic_on_cpu(monkeypatch, golden_dir, F_, guidance):
    r = own_sampler_clip(monkeypatch, golden_dir, F_, guidance)
    out, seen, never, ref_out, g, size = r.out, r.seen, r.never, r.ref_out, r.golden, r.size
    # the reference's callback sees the shadowed loop variable (pipeline :503-510, :556-561): the index of the last context
    # batch at every step - pinned against the reference's own pipeline file in tests/test_dropin_cpu.py
    nwin = 1 if F_ == 1 else 2
    assert seen == [(nwin - 1, t, (1, 4, F_, size // 8, size // 8)) for t in (999, 499)]
    assert len(never) == (1 if nwin == 1 else 0)  # (nwin - 1) % 2: 0 -> called, 1 -> never
    vid = out["videos"]
    assert vid.shape == (1, 3, F_, size, size)
    if F_ == 1:
        want = g["videos"].float()
        err = float((vid[:, :, :, ::8, ::8] - want).norm() / want.norm())
        assert err < 2e-3, err  # the fixture is stored in fp16
        assert float((out["latents"] - g["latents"].float()).norm() / g["latents"].float().norm()) < 2e-3
    else:
        err = float((out["latents"] - ref_out["latents"]).norm() / ref_out["latents"].norm())
        assert err < 1e-4, err  # fp32 both sides: only summation-order noise
        assert float((vid.float() - ref_out["videos"]).norm() / ref_out["videos"].norm()) < 1e-4
