"""Test infrastructure shared by tests/test_dropin_cpu.py, tests/test_pipeline_plumbing_cpu.py and the script that
records their fixtures from the reference (oracle/gen_dropin_golden.py): oracle-backed engine stand-ins, the facade
models and inputs of the recorded clips, and the record / replay of facade calls.

A facade-call trace is a list of calls {"obj", "method", "args", "kwargs", "out"} on this repo's module facades, made by
the reference's own pipeline file. Tensor arguments are stored as descriptors that the replay resolves against a pool of
earlier tensors (every resolved argument and every call's output), so that the large ones - pose features, the UNet's
input windows - are not stored but rebuilt from what the replay itself computed:
  {"raw": key}                stored array                   {"pool": key}           an earlier tensor
  {"scale": key, "by": s}     pool[key] * s                  {"frame": d, "f": i}    resolve(d)[:, :, i]
  {"rep": d, "r": r}          resolve(d) repeated r times along dim 0
  {"frames": [d, ...]}        resolve(d)s stacked along dim 2 (frames)
  {"cat1": [d, ...]}          resolve(d)s concatenated along dim 1 (channels)
  {"inline": values, "dtype": name}   a small tensor written out
Outputs are stored as their shape, the attribute path to the tensor the pipeline uses (".latent_dist.mean", ".sample",
"[0]", ".prev_sample") and a strided sample of its values."""
from __future__ import annotations

import json
from pathlib import Path
from types import SimpleNamespace

import numpy as np
import torch

SCALES = (0.18215, 1 / 0.18215)  # the VAE latent scale, as the pipeline applies it (x * 0.18215, 1 / 0.18215 * x)
OUT_SAMPLE = 32                  # values stored per call output
TRACE_CASES = [(1, 256), (26, 64)]  # BASELINE config 1 (1 frame, 256x256) and 26 frames at 64x64 (two context windows)
STEPS, GUIDANCE, WIDTHS = 2, 3.5, (128, 256, 512, 512)
MOTION_KW = dict(num_attention_heads=8, num_transformer_block=1, attention_block_types=["Temporal_Self", "Temporal_Self"],
                 temporal_position_encoding=True, temporal_position_encoding_max_len=32, temporal_attention_dim_div=1)


class Patch:
    """setattr with undo (what the stand-ins need of pytest's monkeypatch)."""

    def __init__(self):
        self._saved = []

    def setattr(self, obj, name, value):
        self._saved.append((obj, name, obj.__dict__.get(name, Patch) if isinstance(obj, type) else getattr(obj, name)))
        setattr(obj, name, value)

    def undo(self):
        for obj, name, old in reversed(self._saved):
            if old is Patch:
                delattr(obj, name)
            else:
                setattr(obj, name, old)
        self._saved = []


def oracle_engines(monkeypatch, O, cfg, vcfg):
    """Stand-ins for the four engine factories, backed by the oracle (fp32, CPU). `monkeypatch` is anything with
    pytest's setattr(obj, name, value)."""
    from mimo_b200 import ops
    from mimo_b200.host import modules as M

    def ncfhw_to_nhwc(src, cpad, dtype, out=None):
        b, c, f, h, w = src.shape
        t = src.permute(0, 2, 3, 4, 1).reshape(b * f * h * w, c).to(dtype)
        return torch.nn.functional.pad(t, (0, cpad - c))

    def nhwc_to_ncfhw(src, b, c, f, h, w, out_dtype=None, out=None):
        return src[:, :c].reshape(b, f, h, w, c).permute(0, 4, 1, 2, 3).contiguous()

    monkeypatch.setattr(ops, "ncfhw_to_nhwc", ncfhw_to_nhwc)
    monkeypatch.setattr(ops, "nhwc_to_ncfhw", nhwc_to_ncfhw)
    monkeypatch.setattr(M._EngineModel, "_require_cuda", lambda self: None)

    class Den:
        def __init__(self, sd):
            self.sd, self.clip_state = sd, None

        def begin_clip(self, ehs, banks, cfg, frames, branches=None):
            self.clip_state = {"ehs": ehs, "banks": banks, "cfg": cfg}

        def set_cross_attn(self, ehs):
            self.clip_state["ehs"] = ehs

        def forward(self, sample, timestep, pose_nhwc):
            b, c, f, h, w = sample.shape
            pose = pose_nhwc.reshape(b, f, h, w, -1).permute(0, 4, 1, 2, 3)
            st = self.clip_state
            # the host layer hands over the conditional half of the banks only (the unconditional half is never read);
            # the oracle restates the reference, which keeps both: fill the unused slot with a copy
            banks = {k: (v if v.shape[0] == b else v.repeat(b, 1, 1)) for k, v in st["banks"].items()}
            return O.denoising_unet(self.sd, sample, int(timestep), st["ehs"], pose, banks, cfg, cfg=st["cfg"])

    class Ref:
        def __init__(self, sd):
            self.sd = sd

        def write_banks(self, latents, ehs, reader):
            return O.reference_unet_banks(self.sd, latents, ehs, cfg)

    class Pose:
        def __init__(self, sd):
            self.sd = sd

        def forward(self, cond):
            y = O.pose_guider(self.sd, cond)  # [b, C, F, h, w]
            return y.permute(0, 2, 3, 4, 1).reshape(-1, y.shape[1])

    class Vae:
        def __init__(self, sd):
            self.sd = sd

        def encode_mean(self, x):
            return O.vae_encode_mean(self.sd, x, vcfg)

        def decode(self, z):
            return O.vae_decode(self.sd, z, vcfg)

    def cached(factory):
        def engine(self):
            if self._engine is None:
                self._engine = factory(self.state_dict())
            return self._engine
        return engine

    monkeypatch.setattr(M.UNet3DConditionModel, "engine", cached(Den))
    monkeypatch.setattr(M.UNet2DConditionModel, "engine", cached(Ref))
    monkeypatch.setattr(M.PoseGuider, "engine", cached(Pose))
    monkeypatch.setattr(M.AutoencoderKL, "engine", cached(lambda sd: (Vae(sd), Vae(sd))))


def make_checkpoints(tmp: Path):
    """Throw-away 'pretrained_weights' in the directory layout run_animate.py reads (tiny widths: files stay small)."""
    from safetensors.torch import save_file
    from transformers import CLIPVisionConfig, CLIPVisionModelWithProjection

    from mimo_b200.host import schema
    widths = (32, 64, 64, 64)
    gen = torch.Generator().manual_seed(0)
    rnd = lambda shapes: {k: torch.randn(s, generator=gen) * 0.02 for k, s in shapes.items()}
    base = tmp / "stable-diffusion-v1-5" / "unet"
    base.mkdir(parents=True)
    (base / "config.json").write_text(json.dumps(dict(
        sample_size=64, in_channels=4, out_channels=4, block_out_channels=list(widths), layers_per_block=2,
        cross_attention_dim=768, attention_head_dim=8, norm_num_groups=32, norm_eps=1e-5)))
    sd15 = rnd(schema.unet_schema(widths, 2, 768, in_channels=4, out_channels=4, motion=False, out_head=True))
    save_file(sd15, str(base / "diffusion_pytorch_model.safetensors"))
    den_full = rnd(schema.unet_schema(widths, 2, 768, in_channels=8, out_channels=4, motion=True, out_head=True))
    torch.save({k: v for k, v in den_full.items() if "motion_modules" in k}, tmp / "motion_module.pth")
    torch.save(den_full, tmp / "denoising_unet.pth")
    torch.save({k: v for k, v in sd15.items() if not k.startswith(("conv_norm_out", "conv_out"))}, tmp / "reference_unet.pth")
    torch.save(rnd(schema.pose_guider_schema(320, 3, (16, 32, 96, 256))), tmp / "pose_guider.pth")
    vae = tmp / "sd-vae-ft-mse"
    vae.mkdir()
    vw = (32, 32, 64, 64)
    (vae / "config.json").write_text(json.dumps(dict(block_out_channels=list(vw), layers_per_block=2, latent_channels=4,
                                                     in_channels=3, out_channels=3, norm_num_groups=32,
                                                     scaling_factor=0.18215)))
    save_file(rnd(schema.vae_schema(vw, 2, 4, 3, 3)), str(vae / "diffusion_pytorch_model.safetensors"))
    CLIPVisionModelWithProjection(CLIPVisionConfig(hidden_size=32, intermediate_size=64, num_hidden_layers=1,
                                                   num_attention_heads=2, image_size=224, patch_size=32,
                                                   projection_dim=768)).save_pretrained(tmp / "image_encoder")


def composite_case():
    """The synthetic clip of the compositing test (seeded): two context windows sharing frames 3 and 4."""
    from PIL import Image
    rng = np.random.RandomState(3)
    W, H, n_frames, overlay = 96, 72, 7, 2
    contexts = [[0, 1, 2, 3, 4], [3, 4, 5, 6]]  # frames 3, 4 are composited twice: cross-fade
    bboxes = [(0, 60, 4, 72), (20, 96, 0, 50)]   # touch different borders: different feather masks
    bk = [Image.fromarray(rng.randint(0, 256, (H, W, 3), dtype=np.uint8)) for _ in range(n_frames)]
    vid = [Image.fromarray(rng.randint(0, 256, (H, W, 3), dtype=np.uint8)) for _ in range(n_frames)]
    occ = [Image.fromarray(np.repeat(rng.randint(0, 256, (H, W, 1), dtype=np.uint8), 3, axis=2)) for _ in range(n_frames)]
    mask_list = [rng.rand(64, 64).astype(np.float32) for _ in range(16)]
    pads, padvs = [], []
    for k, ctx in enumerate(contexts):
        w_min, w_max, h_min, h_max = bboxes[k]
        bw, bh = w_max - w_min, h_max - h_min
        side = max(bw, bh)
        side += (16 - side % 16) % 16
        top = (side - bh) // 2
        left = (side - bw) // 2
        for _ in ctx:
            pads.append([side, side])
            padvs.append([top, side - bh - top, left, side - bw - left])
    video = torch.rand(3, sum(len(c) for c in contexts), 64, 64, generator=torch.Generator().manual_seed(3))
    return SimpleNamespace(n_frames=n_frames, overlay=overlay, contexts=contexts, bboxes=bboxes, bk=bk, vid=vid, occ=occ,
                           mask_list=mask_list, pads=pads, padvs=padvs, video=video)


def trace_case(F_: int, size: int):
    """Facade models (seeded oracle weights) and PIL inputs of one recorded clip. The images are blocky, so that the
    stored image tensors compress, and not flat: on a constant image GroupNorm divides rounding noise by sqrt(eps)."""
    import PIL.Image
    from transformers import CLIPVisionConfig, CLIPVisionModelWithProjection

    from mimo_b200.host import modules as M
    from mimo_b200.host.scheduler import DDIMScheduler
    from oracle import torch_oracle as O
    seed, vae_widths = 400 + F_, (128, 256, 512, 512) if F_ == 1 else (32, 64, 128, 128)
    cfg, vcfg = O.UNetConfig(block_out_channels=WIDTHS), O.VAEConfig(block_out_channels=vae_widths)
    den = M.UNet3DConditionModel(block_out_channels=WIDTHS, cross_attention_dim=768, use_inflated_groupnorm=True,
                                 use_motion_module=True, motion_module_mid_block=True, motion_module_type="Vanilla",
                                 motion_module_kwargs=MOTION_KW, unet_use_cross_frame_attention=False,
                                 unet_use_temporal_attention=False)
    ref = M.UNet2DConditionModel(block_out_channels=WIDTHS, cross_attention_dim=768)
    pg = M.PoseGuider(WIDTHS[0], conditioning_channels=3, block_out_channels=(16, 32, 96, 256))
    vae = M.AutoencoderKL(block_out_channels=vae_widths)
    sds = dict(den=O.make_denoising_unet_sd(cfg, seed), ref=O.make_reference_unet_sd(cfg, seed + 1),
               pg=O.make_pose_guider_sd(seed + 2, WIDTHS[0]), vae=O.make_vae_sd(vcfg, seed + 3))
    for m, k in ((den, "den"), (ref, "ref"), (pg, "pg"), (vae, "vae")):
        m.load_state_dict(sds[k], strict=True)
    torch.manual_seed(seed + 4)
    clip = CLIPVisionModelWithProjection(CLIPVisionConfig(hidden_size=64, intermediate_size=128, num_hidden_layers=2,
                                                          num_attention_heads=4, image_size=224, patch_size=32,
                                                          projection_dim=768)).eval()
    sched = DDIMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", clip_sample=False,
                          steps_offset=1, prediction_type="v_prediction", rescale_betas_zero_snr=True,
                          timestep_spacing="trailing")
    rng = np.random.RandomState(seed)
    blocky = lambda: PIL.Image.fromarray(np.kron(rng.randint(0, 256, (8, 8, 3)), np.ones((size // 8, size // 8, 1))).astype(np.uint8))
    ref_img, bk = blocky(), blocky()
    poses, bks = [], []
    for i in range(F_):
        a = np.zeros((size, size, 3), np.uint8)
        a[size // 4 + i % 8: size // 2 + i % 8, size // 3: size // 3 + size // 8] = rng.randint(11, 256, 3)
        poses.append(PIL.Image.fromarray(a))
        bks.append(bk)  # animate mode: one background for every frame
    return SimpleNamespace(models=dict(vae=vae, refu=ref, den=den, pg=pg, sched=sched), clip=clip, cfg=cfg, vcfg=vcfg,
                           ref_img=ref_img, poses=poses, bks=bks, size=size, F=F_)


def out_path(out):
    """The attribute path to the tensor the pipeline file reads from a facade call's result, or None."""
    if torch.is_tensor(out):
        return ""
    if isinstance(out, tuple) and out and torch.is_tensor(out[0]):
        return "[0]"
    for p in (".latent_dist.mean", ".sample", ".prev_sample"):
        try:
            v = out
            for a in p.split(".")[1:]:
                v = getattr(v, a)
        except AttributeError:
            continue
        if torch.is_tensor(v):
            return p
    return None


def follow(out, path: str):
    if path == "[0]":
        return out[0]
    for a in path.split(".")[1:]:
        out = getattr(out, a)
    return out


def out_sample(t: torch.Tensor) -> torch.Tensor:
    flat = t.detach().float().reshape(-1)
    return flat[::max(1, flat.numel() // OUT_SAMPLE)][:OUT_SAMPLE].clone()


class Describer:
    """Record side: expresses an argument tensor through the pool of earlier tensors, else stores it."""

    def __init__(self):
        self.pool, self.arrays = {}, {}

    def add(self, key, t):
        self.pool[key] = t.detach().clone()

    def _bases(self, shape_ok):
        for k, p in self.pool.items():
            if shape_ok(p):
                yield {"pool": k}, p
                for s in SCALES:
                    yield {"scale": k, "by": s}, p * s

    def _frame4(self, x):  # a 4-D tensor: an earlier tensor (scaled) or one frame of an earlier 5-D tensor
        for d, p in self._bases(lambda p: p.dim() == 4 and p.shape == x.shape):
            if torch.equal(p, x):
                return d
        for d, p in self._bases(lambda p: p.dim() == 5 and p.shape[:2] == x.shape[:2] and p.shape[3:] == x.shape[2:]):
            for i in range(p.shape[2]):
                if torch.equal(p[:, :, i], x):
                    return {"frame": d, "f": i}
        return None

    def _derive(self, x, split=True):
        if x.dim() not in (4, 5):
            return None
        for d, p in self._bases(lambda p: p.shape == x.shape):
            if torch.equal(p, x):
                return d
        n = x.shape[0]
        for r in range(n, 1, -1):  # repeated along the batch (the CFG pair)
            if n % r == 0 and torch.equal(x[: n // r].repeat(r, *[1] * (x.dim() - 1)), x):
                d = self._derive(x[: n // r])
                return None if d is None else {"rep": d, "r": r}
        if x.dim() == 4:
            return self._frame4(x)
        fr = [self._frame4(x[:, :, j]) for j in range(x.shape[2])]
        if all(f is not None for f in fr):
            return {"frames": fr}
        for c in sorted({p.shape[1] for p in self.pool.values() if p.dim() == 5 and p.shape[1] < x.shape[1]}) if split else ():
            a, b = self._derive(x[:, :c], False), self._derive(x[:, c:], False)
            if a is not None and b is not None:
                return {"cat1": [a, b]}
        return None

    def tensor(self, x):
        x = x.detach()
        if x.numel() <= 16:
            return {"inline": x.reshape(-1).tolist(), "shape": list(x.shape), "dtype": str(x.dtype).removeprefix("torch.")}
        d = next(({"pool": k} for k, p in self.pool.items() if p.shape == x.shape and torch.equal(p, x)), None)
        d = d or self._derive(x)
        if d is None:
            key = f"r{len(self.arrays)}"
            self.arrays[key] = x.numpy().copy()
            self.add(key, x)
            d = {"raw": key}
        return d


def resolve(d, pool, arrays):
    """Replay side: the tensor a descriptor stands for."""
    if "raw" in d:
        if d["raw"] not in pool:
            pool[d["raw"]] = torch.from_numpy(arrays[d["raw"]])
        return pool[d["raw"]]
    if "inline" in d:
        return torch.tensor(d["inline"], dtype=getattr(torch, d["dtype"])).reshape(d["shape"])
    if "pool" in d:
        return pool[d["pool"]]
    if "scale" in d:
        return pool[d["scale"]] * d["by"]
    if "frame" in d:
        return resolve(d["frame"], pool, arrays)[:, :, d["f"]]
    if "rep" in d:
        x = resolve(d["rep"], pool, arrays)
        return x.repeat(d["r"], *[1] * (x.dim() - 1))
    if "frames" in d:
        return torch.stack([resolve(f, pool, arrays) for f in d["frames"]], dim=2)
    return torch.cat([resolve(p, pool, arrays) for p in d["cat1"]], dim=1)


def load_trace(golden_dir: Path, F_: int):
    """The recorded calls of one clip and its arrays (raw arguments "r<n>", output samples "s<k>")."""
    rec = json.loads((golden_dir / "dropin_facade_trace.json").read_text())[str(F_)]
    with np.load(golden_dir / "dropin_facade_trace.npz") as z:
        arrays = {k.split("_", 1)[1]: z[k] for k in z.files if k.startswith(f"c{F_}_")}
    return rec, arrays
