"""Drop-in boundary proof (SURVEY.md §8b) against the reference's own, UNMODIFIED files, on CPU. The reference is not
part of this repository: oracle/gen_dropin_golden.py runs its files over this repo's module facades and stores what they
did under tests/golden/; the tests below hold this repo's code to those recordings. There is no GPU here and the product
has no CPU path, so the facades' engines are replaced - in these tests only - by oracle-backed stand-ins
(oracle/dropin.py).

1. `src/pipelines/pipeline_pose2vid_long_edit_bkfill_roiclip.py`, loaded verbatim with its `src.*` imports resolved to
   THIS repo's overlay (`src/`), ran its Pose2VideoPipeline over the module facades and scheduler for BASELINE config 1
   and a 26-frame two-window clip. Every call it made on them - `UNet3DConditionModel(sample, t,
   encoder_hidden_states=..., pose_cond_fea=..., return_dict=False)[0]`, `PoseGuider(...)`, `AutoencoderKL.encode(...)
   .latent_dist.mean` / `.decode(...).sample`, `UNet2DConditionModel(...)`, `ReferenceAttentionControl(...)`, `.update`,
   `.clear`, `DDIMScheduler.set_timesteps / scale_model_input / step(...).prev_sample` - is in
   tests/golden/dropin_facade_trace.*; the calls are replayed here through the facades and must return what they
   returned. The clips it produced (tests/golden/dropin_pipeline.pt) must also come out of this repo's own sampler.
2. run_animate.py's model-construction block (MIMO.__init__, :60-129), executed statement by statement over the facades
   against throw-away checkpoints (the only edit: the device literal "cuda" -> "cpu"), made the calls recorded in
   tests/golden/run_animate_init_trace.json (`AutoencoderKL.from_pretrained`, `UNet2DConditionModel.from_pretrained`,
   `UNet3DConditionModel.from_pretrained_2d` with the reference's configs/inference/inference_v2.yaml values,
   `PoseGuider(...)`, `DDIMScheduler(**kwargs)`, `load_state_dict`, `Pose2VideoPipeline(...).to(...)`). They are
   replayed here, in order, and must build the same pipeline.
3. run_edit.py's scene-compositing loop and src/pipelines/utils.py: their outputs on seeded inputs."""
import hashlib
import importlib
import json
from pathlib import Path
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle.dropin import (TRACE_CASES, composite_case, follow, load_trace, make_checkpoints, oracle_engines, out_sample,
                           resolve, trace_case)


@pytest.mark.parametrize("F_,size", TRACE_CASES)
def test_reference_pipeline_facade_calls_replay(monkeypatch, golden_dir, F_, size):
    """Every facade call the reference's pipeline file made, in its order, with its arguments (large ones rebuilt from
    what the replay computed before), through the facades: each must return the same structure, shape and values."""
    from mimo_b200.host import modules as M
    from oracle import torch_oracle as O
    rec, arrays = load_trace(golden_dir, F_)
    c = trace_case(F_, size)
    oracle_engines(monkeypatch, O, c.cfg, c.vcfg)
    objs, pool, made = dict(c.models), {}, set()

    def dec(v):
        if isinstance(v, list):
            return [dec(x) for x in v]
        if not isinstance(v, dict):
            return v
        if "tensor" in v:
            return resolve(v["tensor"], pool, arrays)
        if "obj" in v:
            return objs[v["obj"]]
        if "device" in v:
            return torch.device(v["device"])
        return torch.Generator()

    with torch.no_grad():
        for k, e in enumerate(rec["calls"]):
            if "extra" in e:  # the initial noise
                pool[f"o{k}"] = resolve(e["extra"], pool, arrays)
                continue
            args, kwargs = dec(e["args"]), {n: dec(v) for n, v in e["kwargs"].items()}
            if e["method"] is None:
                out = objs[f"rac{k}"] = M.ReferenceAttentionControl(*args, **kwargs)
            else:
                out = getattr(objs[e["obj"]], e["method"])(*args, **kwargs)
            made.add((e["obj"], e["method"]))
            if "out" not in e:
                continue
            got = follow(out, e["out"]["path"])
            assert list(got.shape) == e["out"]["shape"], (k, e["obj"], e["method"])
            s, want = torch.from_numpy(out_sample(got).numpy()), torch.from_numpy(arrays[f"s{k}"])
            assert float((s - want).norm()) <= 1e-4 * float(want.norm()) + 1e-6, (k, e["obj"], e["method"], s, want)
            pool[f"o{k}"] = got
    assert {("den", "__call__"), ("refu", "__call__"), ("pg", "__call__"), ("vae", "encode"), ("vae", "decode"),
            ("sched", "step"), ("sched", "scale_model_input"), ("sched", "set_timesteps")} <= made
    assert {m for o, m in made if o.startswith("rac")} == {"update", "clear"}
    assert c.models["den"]._engine.clip_state is None  # reference_control_reader.clear() reached the engine


@pytest.mark.parametrize("F_,guidance", [(1, 3.5), (26, 3.5), (26, 1.0)])
def test_reference_pipeline_file_runs_over_the_facades(monkeypatch, golden_dir, F_, guidance):
    """The clip (sampled every `stride` pixels), its mean and the callbacks the reference's pipeline file produced over
    the facades (tests/golden/dropin_pipeline.pt), against this repo's sampler on the same models and inputs and against
    the oracle. The facade calls of that run are replayed by test_reference_pipeline_facade_calls_replay."""
    from test_pipeline_plumbing_cpu import own_sampler_clip

    from mimo_b200.host import context
    from mimo_b200.host import modules as M
    want = torch.load(golden_dir / "dropin_pipeline.pt")
    # the pipeline file's intra-package imports land on this repo's overlay
    for mod, names in want["imports"]:
        for n in names:
            assert hasattr(importlib.import_module(mod), n), (mod, n)
    assert importlib.import_module("src.models.mutual_self_attention").ReferenceAttentionControl is M.ReferenceAttentionControl
    assert importlib.import_module("src.pipelines.context").get_context_scheduler is context.get_context_scheduler
    w = want["cases"][f"{F_}-{guidance}"]
    r = own_sampler_clip(monkeypatch, golden_dir, F_, guidance)
    # the callback sees the inner loop's shadowed variable (:503-510): the index of the last context batch, at every step
    assert [(i, t) for i, t, _ in r.seen] == w["seen"] == [(0 if F_ == 1 else 1, 999), (0 if F_ == 1 else 1, 499)]
    assert len(r.never) == w["never"]  # callback_steps = 2: called only where the last batch index is even
    s, gv = w["stride"], w["videos"]
    vid = r.out["videos"].float()
    assert vid.shape == tuple(w["shape"])
    err = float((vid[:, :, :, ::s, ::s] - gv).norm() / gv.norm())
    assert err < 1e-4, err  # fp32 both sides
    assert abs(float(vid.mean()) - w["videos_mean"]) < 1e-5
    if F_ == 1:
        g = torch.load(golden_dir / "pipeline_cfg1.pt")  # the same clip from the reference's own modules
        gc = g["videos"].float()[:, :, :, ::s // 8, ::s // 8]  # stored every 8 pixels
        assert float((gv - gc).norm() / gc.norm()) < 2e-3  # stored in fp16
        assert abs(w["videos_mean"] - g["videos_mean"]) < 1e-4
    else:
        want_o = r.ref_out["videos"][:, :, :, ::s, ::s]
        err = float((gv - want_o).norm() / want_o.norm())
        assert err < 1e-4, err
    assert r.den._engine.clip_state is None  # reference_control_reader.clear() reached the engine


def _replay(trace, names, tmp: Path):
    """Makes the recorded calls in order: `target` is a name in `names` or "$k", the result of call k."""
    got = []

    def dec(v):
        if isinstance(v, list):
            return [dec(x) for x in v]
        if not isinstance(v, dict):
            return v
        if "ref" in v:
            return got[v["ref"]]
        if "path" in v:
            return str(tmp / v["path"])
        if "dtype" in v:
            return getattr(torch, v["dtype"])
        if "tuple" in v:
            return tuple(dec(v["tuple"]))
        return {k: dec(x) for k, x in v["dict"].items()}

    for e in trace:
        t = e["target"]
        obj = got[int(t[1:])] if t.startswith("$") else names[t]
        fn = obj if e["attr"] is None else getattr(obj, e["attr"])
        got.append(fn(*dec(e["args"]), **{k: dec(x) for k, x in e["kwargs"].items()}))
    return got


def test_run_animate_model_construction_block(tmp_path, golden_dir):
    from transformers import CLIPVisionModelWithProjection

    from mimo_b200.host import modules as M
    from mimo_b200.host.pipeline import Pose2VideoPipeline
    from mimo_b200.host.scheduler import DDIMScheduler
    make_checkpoints(tmp_path)
    rec = json.loads((golden_dir / "run_animate_init_trace.json").read_text())
    names = {"AutoencoderKL": M.AutoencoderKL, "DDIMScheduler": DDIMScheduler, "PoseGuider": M.PoseGuider,
             "UNet2DConditionModel": M.UNet2DConditionModel, "UNet3DConditionModel": M.UNet3DConditionModel,
             "CLIPVisionModelWithProjection": CLIPVisionModelWithProjection, "Pose2VideoPipeline": Pose2VideoPipeline,
             "torch.load": torch.load}
    assert {e["target"] for e in rec["calls"] if not e["target"].startswith("$")} <= set(names)
    got = _replay(rec["calls"], names, tmp_path)
    me = SimpleNamespace(pipe=got[rec["self"]["pipe"]["ref"]], width=rec["self"]["width"], height=rec["self"]["height"])
    pipe = me.pipe
    assert isinstance(pipe, Pose2VideoPipeline) and (me.width, me.height) == (512, 512)
    assert pipe.denoising_unet.dtype == torch.float16 and pipe.reference_unet.dtype == torch.float16
    assert pipe.scheduler.config.prediction_type == "v_prediction" and pipe.vae_scale_factor == 8
    # from_pretrained_2d zero-padded conv_in 4 -> 8 input channels, then denoising_unet.pth overwrote it (strict=False)
    want = torch.load(tmp_path / "denoising_unet.pth")["conv_in.weight"].half()
    assert torch.equal(pipe.denoising_unet.state_dict()["conv_in.weight"], want)
    assert "down_blocks.0.motion_modules.0.temporal_transformer.proj_in.weight" in pipe.denoising_unet.state_dict()
    # the models must be the pipeline's: the construction block never rebinds them
    assert pipe.pose_guider is got[next(i for i, e in enumerate(rec["calls"]) if e["target"] == "PoseGuider")]
    # on the CPU the first forward must fail loudly, never fall back to a CPU path
    from mimo_b200.lib import MimoError
    with pytest.raises(MimoError):
        pipe.pose_guider(torch.zeros(1, 3, 1, 64, 64, dtype=torch.float16))


def test_scene_compositing_matches_the_reference_loop(monkeypatch, golden_dir):
    """run_edit.py's post-processing loop (:253-304) with tools/util.py's own get_mask composited composite_case(), with
    and without an occlusion mask (tests/golden/run_edit_composite.json: SHA-256 and sum of every frame); here
    mimo_b200.host.composite.composite_clip runs on the same clip. The blend kernel needs a GPU, so here (and only here)
    ops.composite_frame is the numpy oracle: this pins the helper's host logic (PIL resize / crop / paste, INTER_AREA
    mask resize, mask placement, cross-fade factor, 16-way mask choice) AND the oracle's arithmetic to the reference's
    code; the kernel is pinned to the oracle bit for bit on the GPU (tests/test_clip_composite_gpu.py)."""
    from mimo_b200 import ops
    from mimo_b200.host import composite
    from oracle.composite_oracle import composite_frame
    c = composite_case()
    want = json.loads((golden_dir / "run_edit_composite.json").read_text())

    def blend_on_cpu(canvas, bkf, mask, *, occ=None, vid=None, prev=None, factor=0.0, out=None):
        f = lambda t: None if t is None else t.cpu().numpy()
        return torch.from_numpy(composite_frame(f(canvas), f(bkf), f(mask), f(occ), f(vid), f(prev), factor))

    monkeypatch.setattr(ops, "composite_frame", blend_on_cpu)
    for key, occ in (("occ", c.occ), ("no_occ", None)):  # without: animate-style templates, run_edit.py:262-265
        got = composite.composite_clip(c.video, c.contexts, c.bboxes, c.bk, c.vid, occ, c.pads, c.padvs, c.mask_list,
                                       c.n_frames, c.overlay, device="cpu")
        assert len(want[key]) == c.n_frames
        for i, w in enumerate(want[key]):
            f = np.ascontiguousarray(got[i], dtype=np.uint8)
            assert list(f.shape) == w["shape"] and hashlib.sha256(f.tobytes()).hexdigest() == w["sha256"], (
                key, i, int(f.sum(dtype=np.int64)) - w["sum"])


def test_overlay_pipeline_utils_equal_the_reference(golden_dir):
    """src/pipelines/utils.py (imported by the reference's pipeline file, dead at interpolation_factor = 1): the overlay's
    registry, linear and slerp against what the reference's own file computed (tests/golden/pipeline_utils.pt), bit for
    bit. slerp reduces over the tensor, and ATen's reduction order follows the SIMD width it dispatches to: the fixture
    records the capability it was written with (AVX512); on a CPU of another capability slerp is held to a few ulp."""
    import src.pipelines.utils as ours
    want = torch.load(golden_dir / "pipeline_utils.pt")
    a, b = want["a"], want["b"]
    same_isa = torch.backends.cpu.get_cpu_capability() == want["cpu_capability"]
    for t in (0.0, 0.25, 0.5, 0.9):
        assert torch.equal(ours.linear(a, b, t), want[f"linear-{t}"])
        for name, v1 in (("slerp", b), ("slerp_parallel", a * 1.0001)):  # nearly parallel: the linear branch
            got, ref = ours.slerp(a, v1, t), want[f"{name}-{t}"]
            assert torch.equal(got, ref) or (not same_isa and torch.allclose(got, ref, rtol=1e-6, atol=1e-7))
    for flag in (True, False):
        ours.set_tensor_interpolation_method(flag)
        assert ours.get_tensor_interpolation_method().__name__ == want[f"method-{flag}"]
