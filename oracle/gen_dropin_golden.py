"""Writes the fixtures of tests/test_dropin_cpu.py by running the reference's own, unmodified files over this repo:

  tests/golden/dropin_facade_trace.{json,npz}  every call its pipeline file's Pose2VideoPipeline makes on this repo's
                                           module facades (oracle-backed engines, fp32, CPU) for BASELINE config 1
                                           and a 26-frame two-window clip (format: oracle/dropin.py)
  tests/golden/dropin_pipeline.pt          the clips that pipeline file produced on the plumbing test's inputs
  tests/golden/run_animate_init_trace.json  every call run_animate.py's MIMO.__init__ makes on the facades, in order
  tests/golden/run_edit_composite.json     run_edit.py's compositing loop (tools/util.py's get_mask) on composite_case():
                                           SHA-256 and sum of every uint8 frame
  tests/golden/pipeline_utils.pt           src/pipelines/utils.py's linear / slerp / registry on seeded tensors

Test infrastructure, needs a checkout of the reference:   python oracle/gen_dropin_golden.py --reference <MIMO checkout>
"""
from __future__ import annotations

import argparse
import ast
import hashlib
import importlib.util
import json
import sys
import tempfile
from pathlib import Path
from types import SimpleNamespace

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
GOLDEN = ROOT / "tests" / "golden"
for p in (ROOT, ROOT / "tests" / "compat", ROOT / "oracle" / "diffusers_shim"):
    sys.path.insert(0, str(p))

from oracle import dropin as D  # noqa: E402
CASES = [(1, 3.5), (26, 3.5), (26, 1.0)]


def load_file(name: str, path: Path):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def facade_trace(ref_mod, F_: int, size: int):
    """Runs the reference's Pose2VideoPipeline over trace_case()'s facades and records every call it makes on them."""
    from mimo_b200.host import modules as M
    from mimo_b200.host.scheduler import DDIMScheduler
    from oracle import torch_oracle as O
    c = D.trace_case(F_, size)
    roles = {id(m): k for k, m in c.models.items()}
    desc, calls, depth = D.Describer(), [], [0]

    def enc(v):
        if torch.is_tensor(v):
            return {"tensor": desc.tensor(v)}
        if id(v) in roles:
            return {"obj": roles[id(v)]}
        if isinstance(v, (list, tuple)):
            return [enc(x) for x in v]
        if isinstance(v, torch.device):
            return {"device": str(v)}
        if isinstance(v, torch.Generator):
            return {"generator": True}
        assert v is None or isinstance(v, (str, int, float, bool)), type(v)
        return v

    def record(obj, method, fn, args, kwargs):
        if depth[0]:  # made by a recorded call itself: replaying the outer call repeats it
            return fn(*args, **kwargs)
        e = {"obj": obj, "method": method, "args": enc(list(args)), "kwargs": {k: enc(v) for k, v in kwargs.items()}}
        k = len(calls)
        calls.append(e)
        depth[0] += 1
        try:
            out = fn(*args, **kwargs)
        finally:
            depth[0] -= 1
        if method is None:
            roles[id(out)] = f"rac{k}"
        path = D.out_path(out)
        if path is not None:
            t = D.follow(out, path)
            e["out"] = {"path": path, "shape": list(t.shape)}
            desc.arrays[f"s{k}"] = D.out_sample(t).numpy()
            desc.add(f"o{k}", t)
        return out

    mp = D.Patch()
    try:
        D.oracle_engines(mp, O, c.cfg, c.vcfg)
        for cls, methods in ((M.AutoencoderKL, ("encode", "decode")), (M.UNet2DConditionModel, ("__call__",)),
                             (M.UNet3DConditionModel, ("__call__",)), (M.PoseGuider, ("__call__",)),
                             (DDIMScheduler, ("set_timesteps", "scale_model_input", "step")),
                             (M.ReferenceAttentionControl, ("update", "clear"))):
            for meth in methods:
                def wrapped(self, *a, _orig=getattr(cls, meth), _meth=meth, **kw):
                    if id(self) not in roles:
                        return _orig(self, *a, **kw)
                    return record(roles[id(self)], _meth, lambda *a2, **kw2: _orig(self, *a2, **kw2), a, kw)
                mp.setattr(cls, meth, wrapped)
        mp.setattr(ref_mod, "ReferenceAttentionControl",
                   lambda *a, **kw: record("ReferenceAttentionControl", None, M.ReferenceAttentionControl, a, kw))
        m = c.models
        pipe = ref_mod.Pose2VideoPipeline(vae=m["vae"], image_encoder=c.clip, reference_unet=m["refu"],
                                          denoising_unet=m["den"], pose_guider=m["pg"], scheduler=m["sched"])
        prepare = pipe.prepare_latents

        def prepare_latents(*a, **kw):  # the initial noise enters the trace as data
            t = prepare(*a, **kw)
            calls.append({"extra": desc.tensor(t)})
            desc.add(f"o{len(calls) - 1}", t)
            return t
        pipe.prepare_latents = prepare_latents
        with torch.no_grad():
            pipe(c.ref_img, c.poses, c.bks, size, size, F_, D.STEPS, D.GUIDANCE, generator=torch.manual_seed(42))
    finally:
        mp.undo()
    raw = sum(a.nbytes for k, a in desc.arrays.items() if k.startswith("r"))
    print(f"facade trace F={F_} {size}x{size}: {len(calls)} calls, {raw >> 10} KiB of stored arguments")
    return {"calls": calls}, desc.arrays


def pipeline_cases(ref: Path) -> dict:
    import PIL.Image
    from transformers import CLIPVisionConfig, CLIPVisionModelWithProjection

    from mimo_b200.host import modules as M
    from mimo_b200.host.scheduler import DDIMScheduler
    from oracle import torch_oracle as O
    pipe_file = ref / "src" / "pipelines" / "pipeline_pose2vid_long_edit_bkfill_roiclip.py"
    ref_mod = load_file("_reference_pipeline_file", pipe_file)
    assert ref_mod.ReferenceAttentionControl is M.ReferenceAttentionControl  # src.* resolved to this repo's overlay
    imports = [[n.module, [a.name for a in n.names]] for n in ast.parse(pipe_file.read_text()).body
               if isinstance(n, ast.ImportFrom) and (n.module or "").startswith("src.")]
    g = torch.load(GOLDEN / "pipeline_cfg1.pt")
    cases = {}
    for F_, guidance in CASES:
        seed, size, steps, vae_widths = g["seed"], g["size"], g["steps"], tuple(g["vae_widths"])
        if F_ != 1:
            seed, size, vae_widths = 300, 64, (32, 64, 128, 128)
        widths = (128, 256, 512, 512)
        cfg, vcfg = O.UNetConfig(block_out_channels=widths), O.VAEConfig(block_out_channels=vae_widths)
        mp = D.Patch()
        try:
            D.oracle_engines(mp, O, cfg, vcfg)
            mk = dict(num_attention_heads=8, num_transformer_block=1, attention_block_types=["Temporal_Self", "Temporal_Self"],
                      temporal_position_encoding=True, temporal_position_encoding_max_len=32, temporal_attention_dim_div=1)
            den = M.UNet3DConditionModel(block_out_channels=widths, cross_attention_dim=768, use_inflated_groupnorm=True,
                                         use_motion_module=True, motion_module_mid_block=True, motion_module_type="Vanilla",
                                         motion_module_kwargs=mk, unet_use_cross_frame_attention=False,
                                         unet_use_temporal_attention=False)
            refu = M.UNet2DConditionModel(block_out_channels=widths, cross_attention_dim=768)
            pg = M.PoseGuider(widths[0], conditioning_channels=3, block_out_channels=(16, 32, 96, 256))
            vae = M.AutoencoderKL(block_out_channels=vae_widths)
            sds = dict(den=O.make_denoising_unet_sd(cfg, seed), ref=O.make_reference_unet_sd(cfg, seed + 1),
                       pg=O.make_pose_guider_sd(seed + 2, widths[0]), vae=O.make_vae_sd(vcfg, seed + 3))
            for m, k in ((den, "den"), (refu, "ref"), (pg, "pg"), (vae, "vae")):
                m.load_state_dict(sds[k], strict=True)
            torch.manual_seed(seed + 4)
            clip = CLIPVisionModelWithProjection(CLIPVisionConfig(hidden_size=64, intermediate_size=128, num_hidden_layers=2,
                                                                  num_attention_heads=4, image_size=224, patch_size=32,
                                                                  projection_dim=cfg.cross_attention_dim)).eval()
            sched = DDIMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", clip_sample=False,
                                  steps_offset=1, prediction_type="v_prediction", rescale_betas_zero_snr=True,
                                  timestep_spacing="trailing")
            pipe = ref_mod.Pose2VideoPipeline(vae=vae, image_encoder=clip, reference_unet=refu, denoising_unet=den,
                                              pose_guider=pg, scheduler=sched)
            rng = np.random.RandomState(seed)
            ref_img = PIL.Image.fromarray(rng.randint(0, 256, (size, size, 3), dtype=np.uint8))
            poses, bks = [], []
            for i in range(F_):
                a = np.zeros((size, size, 3), np.uint8)
                a[size // 4: size // 2 + i % 8, size // 3: size // 3 + 40] = rng.randint(11, 256, 3)
                poses.append(PIL.Image.fromarray(a))
                bks.append(PIL.Image.fromarray(rng.randint(0, 256, (size, size, 3), dtype=np.uint8)))
            seen, never = [], []
            with torch.no_grad():
                vid = pipe(ref_img, poses, bks, size, size, F_, steps, guidance, generator=torch.manual_seed(42),
                           callback=lambda i, t, lat: seen.append((i, int(t))), callback_steps=1).videos
                pipe(ref_img, poses, bks, size, size, F_, 1, guidance, generator=torch.manual_seed(42),
                     callback=lambda *a: never.append(a), callback_steps=2)
            assert den._engine.clip_state is None
        finally:
            mp.undo()
        stride = 16  # keeps the fixture small
        cases[f"{F_}-{guidance}"] = {"seen": seen, "never": len(never), "shape": list(vid.shape), "stride": stride,
                                     "videos": vid[:, :, :, ::stride, ::stride].float().clone(),
                                     "videos_mean": float(vid.mean())}
        print(f"pipeline F={F_} guidance={guidance}: callbacks {seen}, mean {float(vid.mean()):.6f}")
    return {"imports": imports, "cases": cases}


class _CudaToCpu(ast.NodeTransformer):
    def visit_Constant(self, node):
        return ast.copy_location(ast.Constant("cpu"), node) if node.value == "cuda" else node


def run_animate_trace(ref: Path, tmp: Path) -> dict:
    """Executes MIMO.__init__ of run_animate.py with every class it constructs from wrapped in a recorder."""
    from omegaconf import OmegaConf  # tests/compat stand-in
    from transformers import CLIPVisionModelWithProjection

    from mimo_b200.host import modules as M
    from mimo_b200.host.pipeline import Pose2VideoPipeline
    from mimo_b200.host.scheduler import DDIMScheduler
    calls, objs = [], {}

    def enc(v):
        if id(v) in objs:
            return {"ref": objs[id(v)]}
        if isinstance(v, torch.dtype):
            return {"dtype": str(v).removeprefix("torch.")}
        if isinstance(v, str) and v.startswith(str(tmp) + "/"):
            return {"path": v[len(str(tmp)) + 1:]}
        if isinstance(v, tuple):
            return {"tuple": [enc(x) for x in v]}
        if isinstance(v, list):
            return [enc(x) for x in v]
        if isinstance(v, dict):
            return {"dict": {k: enc(x) for k, x in v.items()}}
        assert v is None or isinstance(v, (str, int, float, bool)), type(v)
        return v

    keep, depth = [], [0]

    def recorded(target, attr, fn):
        def call(*args, **kwargs):
            if depth[0]:  # made by a recorded call itself (Pipeline.to moving its modules): replaying repeats it
                return fn(*args, **kwargs)
            calls.append({"target": target, "attr": attr, "args": enc(list(args)), "kwargs": enc(kwargs)["dict"]})
            k = len(calls) - 1
            depth[0] += 1
            try:
                out = fn(*args, **kwargs)
            finally:
                depth[0] -= 1
            objs[id(out)] = k
            keep.append(out)  # keeps id() unique
            return out
        return call

    class Rec:
        def __init__(self, name, real):
            self._name, self._real = name, real

        def __call__(self, *a, **kw):
            return recorded(self._name, None, self._real)(*a, **kw)

        def __getattr__(self, attr):
            return recorded(self._name, attr, getattr(self._real, attr))

    D.make_checkpoints(tmp)
    cfg_file = tmp / "animation_edit.yaml"
    cfg_file.write_text("\n".join([
        f'pretrained_base_model_path: "{tmp / "stable-diffusion-v1-5"}"', f'pretrained_vae_path: "{tmp / "sd-vae-ft-mse"}"',
        f'image_encoder_path: "{tmp / "image_encoder"}"', f'denoising_unet_path: "{tmp / "denoising_unet.pth"}"',
        f'reference_unet_path: "{tmp / "reference_unet.pth"}"', f'pose_guider_path: "{tmp / "pose_guider.pth"}"',
        f'motion_module_path: "{tmp / "motion_module.pth"}"',
        f'inference_config: "{ref / "configs" / "inference" / "inference_v2.yaml"}"', "weight_dtype: 'fp16'"]))
    tree = ast.parse((ref / "run_animate.py").read_text())
    init = next(f for c in tree.body if isinstance(c, ast.ClassDef) and c.name == "MIMO"
                for f in c.body if isinstance(f, ast.FunctionDef) and f.name == "__init__")
    body = ast.Module(body=[_CudaToCpu().visit(st) for st in init.body], type_ignores=[])
    ast.fix_missing_locations(body)
    args = SimpleNamespace(config=str(cfg_file), W=512, H=512, seed=42, assets_dir=str(tmp))

    class Torch:  # torch with torch.load recorded
        load = staticmethod(recorded("torch.load", None, torch.load))

        def __getattr__(self, n):
            return getattr(torch, n)

    # method calls on returned objects (.to, .load_state_dict) are recorded by patching them on the classes involved
    import os
    mp = D.Patch()
    try:
        for cls in (M.AutoencoderKL, M.UNet2DConditionModel, M.UNet3DConditionModel, M.PoseGuider,
                    CLIPVisionModelWithProjection, Pose2VideoPipeline):
            for meth in ("to", "load_state_dict"):
                if not hasattr(cls, meth):
                    continue
                orig = getattr(cls, meth)

                def wrapped(self, *a, _orig=orig, _meth=meth, **kw):
                    if id(self) not in objs:
                        return _orig(self, *a, **kw)
                    return recorded(f"${objs[id(self)]}", _meth, lambda *a2, **kw2: _orig(self, *a2, **kw2))(*a, **kw)
                mp.setattr(cls, meth, wrapped)
        ns = dict(torch=Torch(), os=os, OmegaConf=OmegaConf, AutoencoderKL=Rec("AutoencoderKL", M.AutoencoderKL),
                  DDIMScheduler=Rec("DDIMScheduler", DDIMScheduler),
                  UNet2DConditionModel=Rec("UNet2DConditionModel", M.UNet2DConditionModel),
                  UNet3DConditionModel=Rec("UNet3DConditionModel", M.UNet3DConditionModel),
                  PoseGuider=Rec("PoseGuider", M.PoseGuider),
                  CLIPVisionModelWithProjection=Rec("CLIPVisionModelWithProjection", CLIPVisionModelWithProjection),
                  Pose2VideoPipeline=Rec("Pose2VideoPipeline", Pose2VideoPipeline), parse_args=lambda: args,
                  load_mask_list=lambda p: [], self=SimpleNamespace(), debug_mode=False)
        exec(compile(body, "run_animate.py:MIMO.__init__", "exec"), ns)
    finally:
        mp.undo()
    me = ns["self"]
    assert isinstance(me.pipe, Pose2VideoPipeline)
    print(f"run_animate.py MIMO.__init__: {len(calls)} calls on the facades")
    return {"calls": calls, "self": {"pipe": enc(me.pipe), "width": me.width, "height": me.height}}


def run_edit_composite(ref: Path) -> dict:
    import cv2
    from PIL import Image
    ref_util = load_file("_reference_tools_util", ref / "tools" / "util.py")
    c = D.composite_case()
    tree = ast.parse((ref / "run_edit.py").read_text())
    run = next(f for k in tree.body if isinstance(k, ast.ClassDef) and k.name == "MIMO"
               for f in k.body if isinstance(f, ast.FunctionDef) and f.name == "run")
    loop = next(st for st in run.body if isinstance(st, ast.For) and isinstance(st.iter, ast.Call)
                and getattr(st.iter.func, "id", "") == "enumerate" and getattr(st.iter.args[0], "id", "") == "context_list")
    init = next(st for st in run.body if isinstance(st, ast.Assign) and getattr(st.targets[0], "id", "") == "res_images")
    idx0 = next(st for st in run.body if isinstance(st, ast.Assign) and getattr(st.targets[0], "id", "") == "video_idx")
    mod = ast.Module(body=[idx0, init, loop], type_ignores=[])
    ast.fix_missing_locations(mod)
    out = {}
    for key, occ in (("occ", c.occ), ("no_occ", None)):
        me = SimpleNamespace(args=SimpleNamespace(L=c.n_frames), mask_list=c.mask_list)
        ns = dict(np=np, cv2=cv2, Image=Image, get_mask=ref_util.get_mask, self=me, context_list=c.contexts,
                  bbox_clip_list=c.bboxes, bk_images_ori=c.bk, vid_images_ori=c.vid, occ_mask_images=occ,
                  clip_pad_list_context=c.pads, clip_padv_list_context=c.padvs, video=c.video, overlay=c.overlay)
        exec(compile(mod, "run_edit.py:MIMO.run[post-process]", "exec"), ns)
        frames = [np.ascontiguousarray(f, dtype=np.uint8) for f in ns["res_images"]]
        out[key] = [{"shape": list(f.shape), "sha256": hashlib.sha256(f.tobytes()).hexdigest(), "sum": int(f.sum(dtype=np.int64))}
                    for f in frames]
    print(f"run_edit.py compositing: {len(out['occ'])} frames per case")
    return out


def pipeline_utils(ref: Path) -> dict:
    r = load_file("_ref_pipeline_utils", ref / "src" / "pipelines" / "utils.py")
    g = torch.Generator().manual_seed(3)
    a, b = torch.randn(4, 8, 8, generator=g), torch.randn(4, 8, 8, generator=g)
    out = {"a": a, "b": b, "cpu_capability": torch.backends.cpu.get_cpu_capability()}
    for t in (0.0, 0.25, 0.5, 0.9):
        out[f"linear-{t}"] = r.linear(a, b, t)
        out[f"slerp-{t}"] = r.slerp(a, b, t)
        out[f"slerp_parallel-{t}"] = r.slerp(a, a * 1.0001, t)
    for flag in (True, False):
        r.set_tensor_interpolation_method(flag)
        out[f"method-{flag}"] = r.get_tensor_interpolation_method().__name__
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", type=Path, required=True, help="root of a MIMO checkout (run_animate.py, src/, ...)")
    ref = ap.parse_args().reference.resolve()
    ref_mod = load_file("_reference_pipeline_file", ref / "src" / "pipelines" / "pipeline_pose2vid_long_edit_bkfill_roiclip.py")
    traces, arrays = {}, {}
    for F_, size in D.TRACE_CASES:
        traces[str(F_)], arr = facade_trace(ref_mod, F_, size)
        arrays.update({f"c{F_}_{k}": v for k, v in arr.items()})
    (GOLDEN / "dropin_facade_trace.json").write_text(json.dumps(traces, separators=(",", ":")) + "\n")
    np.savez_compressed(GOLDEN / "dropin_facade_trace.npz", **arrays)
    torch.save(pipeline_cases(ref), GOLDEN / "dropin_pipeline.pt")
    with tempfile.TemporaryDirectory() as tmp:
        trace = run_animate_trace(ref, Path(tmp).resolve())
    (GOLDEN / "run_animate_init_trace.json").write_text(json.dumps(trace, indent=1) + "\n")
    (GOLDEN / "run_edit_composite.json").write_text(json.dumps(run_edit_composite(ref), indent=1) + "\n")
    torch.save(pipeline_utils(ref), GOLDEN / "pipeline_utils.pt")


if __name__ == "__main__":
    main()
