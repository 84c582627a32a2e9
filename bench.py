#!/usr/bin/env python
"""bench.py — frames/sec of the MIMO denoising path on B200 (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--dump-outputs DIR]   our engine (one JSON line on rank 0)
  python bench.py --impl reference [--gpus N] --steps K --warmup W   the oracle port on the host cores

Workload (BASELINE.json configs[1]): 512x512, 24 frames, 20 DDIM steps, CFG 3.5, fp16, synthetic PIL inputs,
seeded random weights of the full architecture (denoising UNet3D 1.31 B params, reference UNet 0.86 B, PoseGuider,
sd-vae-ft-mse-shaped VAE, CLIP ViT-L/14 vision tower) — there are no checkpoints or assets offline.

A "step" is one whole clip: Pose2VideoPipeline's work from CLIP/VAE-encode/pose/reference-UNet through 20 denoising
steps to the batched VAE decode. `value` times sample_tensors() with every input already in HBM; `e2e` times the
public __call__ (PIL in -> CPU video tensor out: PIL pre-processing, pinned H2D, D2H of the clip inside the timed
region). Inputs differ per step by the noise seed (pre-generated, resident in HBM); the UNet touches > 2.6 GB of
weights + multi-hundred-MB activations per forward, far beyond the 126 MB L2, so no explicit L2 flush is needed
between steps.

Both arms print the same `config`. The reference arm times the oracle port (the reference's PyTorch graph, fp32) on the
host cores: every step is a BOUNDED sample of the workload — one CFG UNet3D forward on f_s of the 24 frames at the full
64x64 latent size, f_s chosen so that warmup + steps fit a few minutes — and `value` extrapolates it to the whole clip
(the formula is in cpu_baseline.sample); `ms_per_step` is the real wall time of a step.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

import numpy as np  # noqa: E402
import torch  # noqa: E402

WIDTH = HEIGHT = 512
FRAMES = 24
DDIM_STEPS = 20
GUIDANCE = 3.5
METRIC = "frames/sec @ 512x512x24f, 20 DDIM steps"
# algorithmic work per output frame at this config (SURVEY.md §8d / BASELINE.md §2)
TFLOP_PER_FRAME = 49.3

CONFIG = {"workload": "512x512 x 24-frame animate, 20 DDIM steps, CFG 3.5, fp16 (BASELINE.json configs[1])",
          "frames": FRAMES, "ddim_steps": DDIM_STEPS, "guidance_scale": GUIDANCE,
          "l2": "inputs/weights per forward >> 126 MB L2; no explicit flush"}
DTYPE, DTYPE_NAME, NOISE_BK = torch.float16, "fp16", False


def select_config(k: int) -> None:
    """BASELINE.json configs[k-1]. 2 (default, also 3 = the same clip on 8 GPUs): the metric's configuration. 4 and 5 are
    extra lines for the 8-GPU node: `bench.py --config 4|5` (TFLOP per output frame from SURVEY.md §8d)."""
    global WIDTH, HEIGHT, FRAMES, DDIM_STEPS, METRIC, TFLOP_PER_FRAME, CONFIG, DTYPE, DTYPE_NAME, NOISE_BK
    if k in (2, 3):
        return
    if k == 4:
        WIDTH = HEIGHT = 768
        FRAMES, DDIM_STEPS, TFLOP_PER_FRAME = 48, 30, 285.7
        DTYPE, DTYPE_NAME = torch.bfloat16, "bf16"
        name = "768x768 x 48-frame animate (3 context windows), 30 DDIM steps, CFG 3.5, bf16 (BASELINE.json configs[3])"
    elif k == 5:
        FRAMES, DDIM_STEPS, TFLOP_PER_FRAME, NOISE_BK = 64, 20, 72.0, True
        name = ("512x512 x 64-frame character edit (4 context windows, a distinct background per frame), 20 DDIM steps, "
                "CFG 3.5, fp16 (BASELINE.json configs[4]); scene compositing is host-side in run_edit.py and not timed")
    else:
        raise SystemExit(f"--config {k}: BASELINE.json has configs 1..5 (1 is the CPU plumbing case: tests/)")
    METRIC = f"frames/sec @ {WIDTH}x{HEIGHT}x{FRAMES}f, {DDIM_STEPS} DDIM steps"
    CONFIG = {"workload": name, "frames": FRAMES, "ddim_steps": DDIM_STEPS, "guidance_scale": GUIDANCE,
              "l2": "inputs/weights per forward >> 126 MB L2; no explicit flush"}

SCHED_KW = dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", clip_sample=False, steps_offset=1,
                prediction_type="v_prediction", rescale_betas_zero_snr=True, timestep_spacing="trailing")
MOTION_KW = dict(num_attention_heads=8, num_transformer_block=1, attention_block_types=["Temporal_Self", "Temporal_Self"],
                 temporal_position_encoding=True, temporal_position_encoding_max_len=32, temporal_attention_dim_div=1)


def synthetic_inputs(frames: int, size: int, seed: int = 0, noise_bk: bool = False):
    """SURVEY.md §8d: seeded uint8 reference image, pose frames = black with a coloured blob, white backgrounds."""
    import PIL.Image
    rng = np.random.RandomState(seed)
    ref_img = PIL.Image.fromarray(rng.randint(0, 256, (size, size, 3), dtype=np.uint8))
    poses, bks = [], []
    for i in range(frames):
        a = np.zeros((size, size, 3), np.uint8)
        a[size // 4 + i: size // 2 + i, size // 3: size // 3 + size // 8] = rng.randint(11, 256, 3)
        poses.append(PIL.Image.fromarray(a))
        bks.append(PIL.Image.fromarray(rng.randint(0, 256, (size, size, 3), dtype=np.uint8) if noise_bk
                                       else np.full((size, size, 3), 255, np.uint8)))
    return ref_img, poses, bks


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        pw = [float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": reasons}


DUMP_BYTES = 60 << 20  # what --dump-outputs may write in all: under 64 MB with the .npy headers


def dump_outputs(outputs: dict, dest: Path) -> None:
    """Writes each output tensor as <dest>/<name>.npy in float32, DUMP_BYTES in all. An output larger than its share of
    what is left is stored as a sample: its elements at the sorted flat indices that torch.randperm draws from a generator
    seeded with 0. The sample depends only on the output's size, so runs with the same arguments store the same
    elements."""
    dest.mkdir(parents=True, exist_ok=True)
    items = sorted(outputs.items(), key=lambda kv: kv[1].numel())
    left = DUMP_BYTES
    for i, (name, t) in enumerate(items):
        flat = t.detach().float().cpu().reshape(-1)
        share = left // (len(items) - i) // 4
        if flat.numel() <= share:
            arr, what = flat.reshape(t.shape).numpy(), "all"
        else:
            idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(0))[:share].sort().values
            arr, what = flat[idx].numpy(), f"{share} seeded flat-index samples"
        np.save(dest / f"{name}.npy", arr)
        left -= arr.nbytes
        print(f"bench.py: {dest / name}.npy <- {name} {tuple(t.shape)}: {what}", file=sys.stderr)


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return d.get("bf16_tflops_sustained", 1439.7), d.get("hbm_gbs", 6566.4), "measured (MEASURED_PEAKS.json, sustained)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


# =====================================================================================================
# our engine
# =====================================================================================================
def build_pipeline(device, rank: int = 0, world: int = 1):
    from transformers import CLIPVisionConfig, CLIPVisionModelWithProjection

    from mimo_b200.host import modules as M
    from mimo_b200.host.pipeline import Pose2VideoPipeline
    from mimo_b200.host.scheduler import DDIMScheduler
    torch.manual_seed(42)  # run_animate.py:46 default seed; weights are the modules' seeded default init
    den = M.UNet3DConditionModel(cross_attention_dim=768, use_inflated_groupnorm=True, use_motion_module=True,
                                 motion_module_mid_block=True, motion_module_type="Vanilla",
                                 motion_module_kwargs=MOTION_KW, unet_use_cross_frame_attention=False,
                                 unet_use_temporal_attention=False)
    ref = M.UNet2DConditionModel(cross_attention_dim=768)
    pg = M.PoseGuider(320, 3, (16, 32, 96, 256))
    vae = M.AutoencoderKL()
    clip = CLIPVisionModelWithProjection(CLIPVisionConfig(hidden_size=1024, intermediate_size=4096, num_hidden_layers=24,
                                                          num_attention_heads=16, image_size=224, patch_size=14,
                                                          projection_dim=768)).eval()
    pipe = Pose2VideoPipeline(vae=vae, image_encoder=clip, reference_unet=ref, denoising_unet=den, pose_guider=pg,
                              scheduler=DDIMScheduler(**SCHED_KW))
    pipe.to(device, dtype=DTYPE)
    if world > 1:
        pipe.enable_frame_sharding(rank, world)
    return pipe


def run_ours(args):
    import torch.distributed as dist

    from mimo_b200 import ops
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    pipe = build_pipeline(device, rank, world)
    ref_img, poses, bks = synthetic_inputs(FRAMES, WIDTH, noise_bk=NOISE_BK)

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def clip_seed(i):
        return torch.Generator().manual_seed(42 + i)

    # ---- device-resident runs (value) ------------------------------------------------------------------
    host = pipe.preprocess(ref_img, poses, bks, WIDTH, HEIGHT, FRAMES, clip_seed(0), DTYPE)
    dev_in = {k: v.to(device) for k, v in host.items()}
    if args.one_clip:
        t0 = time.perf_counter()
        pipe.sample_tensors(dev_in, DDIM_STEPS, GUIDANCE)
        sync()
        if rank == 0:
            print(json.dumps({"one_clip_s": round(time.perf_counter() - t0, 3), "note": "profiling aid, not a bench value"}))
        return
    # one noise tensor per step, drawn like prepare_latents does (CPU generator, fp16) and resident before timing
    lat_shape = tuple(host["latents"].shape)
    seeds = [torch.randn(lat_shape, generator=clip_seed(1000 + i), dtype=DTYPE).to(device)
             for i in range(args.steps)]
    for i in range(args.warmup):
        pipe.sample_tensors(dev_in, DDIM_STEPS, GUIDANCE)
    sync()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = ops.launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync()
    e0.record()
    for i in range(args.steps):
        out = pipe.sample_tensors({**dev_in, "latents": seeds[i]}, DDIM_STEPS, GUIDANCE)
    e1.record()
    sync()
    ms = e0.elapsed_time(e1)
    launches = ops.launches() - l0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:  # after the clock sampler: the dump keeps the GPU idle for seconds
        dump_outputs(out, Path(args.dump_outputs))
    pipe._collect_timings()
    phases = dict(pipe.timings)
    if world > 1:
        t = torch.tensor([ms], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t)
    ms_per_step = ms / args.steps
    value = FRAMES / (ms_per_step / 1e3)

    # ---- end to end through the public API (PIL in, CPU tensor out) -------------------------------------
    # warm the host path: two untimed calls whose results are both alive, as `res` and the clip being produced are in the
    # timed loop below, so the pinned-memory cache holds the two result buffers before timing starts
    warm = [pipe(ref_img, poses, bks, WIDTH, HEIGHT, FRAMES, DDIM_STEPS, GUIDANCE, generator=clip_seed(98 + i))
            for i in range(2)]
    res = warm.pop()
    del warm
    sync()
    k_e2e = args.steps
    t0 = time.perf_counter()
    for i in range(k_e2e):
        res = pipe(ref_img, poses, bks, WIDTH, HEIGHT, FRAMES, DDIM_STEPS, GUIDANCE, generator=clip_seed(i))
    sync()
    e2e_s = (time.perf_counter() - t0) / k_e2e
    if world > 1:
        t = torch.tensor([e2e_s], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t)
    assert res.videos.shape == (1, 3, FRAMES, HEIGHT, WIDTH)

    roofline, calls, kernels, kernels_src = None, None, None, "skipped (--no-breakdown)"
    if not args.no_breakdown:
        try:
            # ---- roofline of the dominant kernel: one extra, untimed clip with CUDA-event brackets around every C-ABI call ----
            # The brackets must time kernels, not the host: each forward is preceded by a ~40 ms device-side spin so that the
            # host runs ahead and the ~1 400 launches of the forward sit back to back in the stream when they execute.
            # (Brackets are exact for long kernels - the GEMM / conv / attention families; they over-read the ~10 us kernels by
            # launch latency, which is why the per-kernel table below comes from CUPTI on a graph-replay clip instead.)
            den_eng = pipe.denoising_unet.engine()
            orig_impl = den_eng._forward_impl

            def queued_impl(*a):
                torch.cuda._sleep(80_000_000)
                return orig_impl(*a)

            den_eng._forward_impl = queued_impl
            ops.PROFILE = []
            pipe.sample_tensors(dev_in, DDIM_STEPS, GUIDANCE)
            torch.cuda.synchronize()
            prof, ops.PROFILE = ops.PROFILE, None
            den_eng._forward_impl = orig_impl
            if args.dump_calls and rank == 0:
                with open(args.dump_calls, "w") as fcsv:
                    fcsv.write("idx,name,flops,bytes,ms\n")
                    for i, (name, fl, by, a, b) in enumerate(prof):
                        fcsv.write(f"{i},{name},{fl:.0f},{by:.0f},{a.elapsed_time(b):.4f}\n")
            agg = {}
            for name, fl, by, a, b in prof:
                d = agg.setdefault(name, [0.0, 0.0, 0.0, 0])
                d[0] += a.elapsed_time(b)
                d[1] += fl
                d[2] += by
                d[3] += 1
            total_ms = sum(d[0] for d in agg.values())
            peak_tf, peak_gbs, peak_src = measured_peaks()
            calls = {}
            for name, (t_ms, fl, by, cnt) in sorted(agg.items(), key=lambda kv: -kv[1][0]):
                calls[name] = {"ms": round(t_ms, 2), "launches": cnt, "tflops": round(fl / t_ms / 1e9, 1) if fl else None,
                               "gbs": round(by / t_ms / 1e6, 1)}
            # The dominant kernel is gemm_tcgen05_kernel: the plain GEMMs ("gemm") and the implicit-GEMM 3x3 convolutions
            # ("conv3x3") are the same kernel template in its two addressing modes.
            fam = {"gemm_tcgen05_kernel": ("gemm", "conv3x3"), "attn_spatial": ("attn_spatial",)}
            fam_ms = {k: sum(agg[n][0] for n in names if n in agg) for k, names in fam.items()}
            others = {n: agg[n][0] for n in agg if not any(n in names for names in fam.values())}
            dname = max({**fam_ms, **others}.items(), key=lambda kv: kv[1])[0]
            members = fam.get(dname, (dname,))
            dms = sum(agg[n][0] for n in members if n in agg)
            dfl = sum(agg[n][1] for n in members if n in agg)
            dby = sum(agg[n][2] for n in members if n in agg)
            dcnt = sum(agg[n][3] for n in members if n in agg)
            tensor_bound = dname in ("gemm_tcgen05_kernel", "attn_spatial")
            achieved = dfl / dms / 1e9 if tensor_bound else dby / dms / 1e6
            peak = peak_tf if tensor_bound else peak_gbs
            # DRAM bytes per launch of this kernel from the committed `ncu --set full` capture of THIS gpu count, else null
            traffic, traffic_src = None, None
            tpath = ROOT / "profiles" / "ncu_traffic.json"
            if tpath.exists():
                ent = json.loads(tpath.read_text()).get(str(world), {}).get(dname)
                if ent:
                    traffic, traffic_src = ent.get("dram_bytes_per_launch"), ent.get("source")
            roofline = {"kernel": dname, "bound": "tensor" if tensor_bound else "hbm", "achieved": round(achieved, 1),
                        "peak": peak, "unit": "TFLOP/s" if tensor_bound else "GB/s", "frac": round(achieved / peak, 4),
                        "traffic": traffic, "traffic_source": traffic_src, "algorithmic_bytes_per_launch": round(dby / dcnt),
                        "peak_source": peak_src, "launches": dcnt, "avg_launch_ms": round(dms / dcnt, 4),
                        "share_of_bracketed_clip": round(dms / total_ms, 4),
                        "whole_path_frac_of_tensor_peak": round(TFLOP_PER_FRAME * value / (world * peak_tf), 4)}

            # ---- per-kernel table: CUPTI kernel records of one more clip executed exactly like the timed ones (graph replay) --
            kernels, kernels_src = None, None
            try:
                from torch.profiler import ProfilerActivity, profile
                with profile(activities=[ProfilerActivity.CUDA]) as tp:
                    sync()  # CUPTI start-up differs per rank: this barrier absorbs the skew, not the clip's first collective
                    pipe.sample_tensors(dev_in, DDIM_STEPS, GUIDANCE)
                    torch.cuda.synchronize()
                rows = {}
                for ev in tp.key_averages():
                    us = getattr(ev, "device_time_total", None)
                    if us is None:
                        us = getattr(ev, "cuda_time_total", 0.0)
                    if us <= 0:
                        continue
                    if "AllReduce" in ev.key:
                        continue  # the barrier above
                    nm = ev.key.replace("void ", "").split("(")[0]
                    nm = nm if len(nm) <= 72 else nm[:72]
                    r = rows.setdefault(nm, [0.0, 0])
                    r[0] += us / 1e3
                    r[1] += ev.count
                tot = sum(v[0] for v in rows.values())
                kernels = {k: {"ms": round(v[0], 2), "share": round(v[0] / tot, 4), "launches": v[1]}
                           for k, v in sorted(rows.items(), key=lambda kv: -kv[1][0])[:24]}
                kernels["_total_kernel_ms"] = round(tot, 1)
                kernels_src = "CUPTI kernel records (torch.profiler) of one extra clip under CUDA-graph replay; not the timed clips"
                fam_cupti = sum(v[0] for k, v in rows.items() if dname.split("_kernel")[0] in k)
                roofline["cupti_ms_per_clip"] = round(fam_cupti, 1)
                roofline["bracket_ms_per_clip"] = round(dms, 1)
            except Exception as ex:  # noqa: BLE001 - the table is a diagnostic; the bench line must not depend on CUPTI
                kernels_src = f"unavailable ({type(ex).__name__}: {ex})"

        except Exception as ex:  # noqa: BLE001 - the breakdown is diagnostic: the measured line above must still print
            ops.PROFILE = None
            eng = pipe.denoising_unet.engine()
            eng.__dict__.pop("_forward_impl", None)  # drop the queued wrapper if it is still installed
            roofline, kernels_src = None, f"breakdown failed ({type(ex).__name__}: {ex})"
    if rank != 0:
        return
    cpu = None
    if not (args.no_cpu_baseline or world > 1):
        try:
            cpu = cpu_baseline_sample(frames=8)
        except Exception as ex:  # noqa: BLE001 - a host-side failure must not cost the measured GPU line
            cpu = {"value": None, "unit": "frames/s", "cores": usable_cores(), "kind": "port",
                   "sample": f"failed: {type(ex).__name__}: {ex}"}
    par = "1 GPU"
    if world > 1:
        from mimo_b200.host.shard import ShardPlan
        from mimo_b200.host.context import uniform
        wins = list(uniform(0, DDIM_STEPS, FRAMES, 24, 1, 4))
        pl = ShardPlan.make(world, 0, True, len(wins), len(wins[0]), min_tokens=(HEIGHT // 64) * (WIDTH // 64))
        par = (f"{world} GPUs = CFG branches x{pl.cfg_ways} * windows x{pl.win_ways} * frames x{pl.frame_ways}; "
               "frames<->pixels exchange over NVLink peer memory (mimo_exchange), no NCCL on the data path")
    line = {
        "metric": METRIC, "value": round(value, 4), "unit": "frames/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(ms_per_step, 2), "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": DTYPE_NAME, "data": "synthetic", "config": dict(CONFIG), "parallelism": par,
        "e2e": {"value": round(FRAMES / e2e_s, 4), "unit": "frames/s", "h2d_bytes_per_step": pipe.io_bytes["h2d"],
                "d2h_bytes_per_step": pipe.io_bytes["d2h"], "clips_timed": k_e2e},
        "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
        "whole_path_frac_of_tensor_peak": round(TFLOP_PER_FRAME * value / (world * measured_peaks()[0]), 4),
        "phases_ms": {k: round(v, 1) for k, v in phases.items()}, "calls_bracketed": calls, "kernels": kernels,
        "kernels_source": kernels_src,
    }
    print(json.dumps(line))


# =====================================================================================================
# CPU baseline: the oracle port of the reference's PyTorch graph on the host cores
# =====================================================================================================
_CPU_WEIGHTS: dict = {}


def usable_cores() -> int:
    """Host threads this process may really use: CPU affinity, capped by a cgroup CPU quota if there is one
    (`os.cpu_count()` reports the machine, not the container)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    for quota_f, period_f in (("/sys/fs/cgroup/cpu.max", None),
                              ("/sys/fs/cgroup/cpu/cpu.cfs_quota_us", "/sys/fs/cgroup/cpu/cpu.cfs_period_us")):
        try:
            if period_f is None:
                q, per = Path(quota_f).read_text().split()
            else:
                q, per = Path(quota_f).read_text().strip(), Path(period_f).read_text().strip()
            if q not in ("max", "-1") and float(per) > 0:
                n = min(n, max(1, int(float(q) / float(per))))
            break
        except (OSError, ValueError):
            continue
    return max(1, n)


def pick_cpu_threads() -> int:
    """The thread count the CPU arm runs with: the fastest of {all usable, 1/2, 1/4} on a one-second probe of the
    UNet's dominant op (a 320-channel 3x3 convolution at the sample's 64x64 resolution). With every hardware thread of
    a 128-thread host on this small a problem the oracle ran 30x slower than with 8 threads - that would be an
    unfairly slow baseline."""
    n = usable_cores()
    x = torch.randn(2, 320, 64, 64)
    w = torch.randn(320, 320, 3, 3)
    cands = sorted({n, max(1, n // 2), max(1, n // 4)}, reverse=True)
    times = {c: float("inf") for c in cands}
    with torch.no_grad():
        for _ in range(2):  # two rounds, best of: the first touches cold pages
            for c in cands:
                torch.set_num_threads(c)
                torch.nn.functional.conv2d(x, w, padding=1)  # warm the primitive cache for this thread count
                t0 = time.perf_counter()
                for _ in range(3):
                    torch.nn.functional.conv2d(x, w, padding=1)
                times[c] = min(times[c], time.perf_counter() - t0)
    best = cands[0]
    for c in cands[1:]:  # prefer more threads unless fewer are clearly (25 %) faster
        if times[c] < 0.75 * times[best]:
            best = c
    return best


def _cpu_setup():
    from oracle import torch_oracle as O
    cfg, vcfg = O.UNetConfig(), O.VAEConfig()
    if not _CPU_WEIGHTS:  # seeded random weights, built once per process (20 s of the first sample otherwise)
        _CPU_WEIGHTS.update(den=O.make_denoising_unet_sd(cfg, 1), ref=O.make_reference_unet_sd(cfg, 2),
                            vae=O.make_vae_sd(vcfg, 4), cores=pick_cpu_threads())
    torch.set_num_threads(_CPU_WEIGHTS["cores"])
    return O, cfg, vcfg


def cpu_fixed_parts(seed: int = 0) -> dict:
    """Once-per-clip pieces of the reference's path on the host: the reference UNet pass (banks), one VAE-decode frame,
    one VAE-encode frame, all at 512x512 / 64x64 latents, fp32. Returns seconds each and the banks."""
    O, cfg, vcfg = _cpu_setup()
    g = torch.Generator().manual_seed(seed)
    h = w = HEIGHT // 8
    ehs = torch.cat([torch.zeros(1, 1, 768), torch.randn(1, 1, 768, generator=g)])
    with torch.no_grad():
        t0 = time.perf_counter()
        banks = O.reference_unet_banks(_CPU_WEIGHTS["ref"], torch.randn(2, 4, h, w, generator=g), ehs, cfg)
        t_ref = time.perf_counter() - t0
        t0 = time.perf_counter()
        O.vae_decode(_CPU_WEIGHTS["vae"], torch.randn(1, 4, h, w, generator=g), vcfg)
        t_dec = time.perf_counter() - t0
        t0 = time.perf_counter()
        O.vae_encode_mean(_CPU_WEIGHTS["vae"], torch.randn(1, 3, HEIGHT, WIDTH, generator=g), vcfg)
        t_enc = time.perf_counter() - t0
    return {"t_ref": t_ref, "t_dec": t_dec, "t_enc": t_enc, "banks": banks, "ehs": ehs}


def cpu_unet_sample(frames: int, fixed: dict, seed: int = 0) -> float:
    """Seconds of ONE CFG forward of the denoising UNet3D on `frames` of the 24 frames at 64x64 latents (fp32, oracle
    port of src/models/unet_3d_edit_bkfill.py:398-576 with banks, pose features and temporal attention over `frames`)."""
    O, cfg, _ = _cpu_setup()
    g = torch.Generator().manual_seed(100 + seed)
    h = w = HEIGHT // 8
    x = torch.randn(2, 8, frames, h, w, generator=g)
    pose = torch.randn(2, 320, frames, h, w, generator=g)
    with torch.no_grad():
        t0 = time.perf_counter()
        O.denoising_unet(_CPU_WEIGHTS["den"], x, 499, fixed["ehs"], pose, fixed["banks"], cfg, cfg=True)
        return time.perf_counter() - t0


def _extrapolate(t_unet: float, frames: int, fx: dict) -> float:
    """Clip seconds from a sample: the UNet forward is linear in frames (exact up to the 24x24 temporal attention,
    0.2 % of the FLOPs); 20 steps; 24 decodes; animate mode encodes 2 distinct images (reference + white background)."""
    return DDIM_STEPS * t_unet * (FRAMES / frames) + FRAMES * fx["t_dec"] + 2 * fx["t_enc"] + fx["t_ref"]


def cpu_baseline_sample(frames: int = 8, seed: int = 0) -> dict:
    """Bounded sample for the engine arm's `cpu_baseline` (about 20-30 s): one CFG UNet3D forward on `frames` of the 24
    frames + the once-per-clip pieces, extrapolated to the clip. A reported baseline, not a target."""
    fx = cpu_fixed_parts(seed)
    t_unet = cpu_unet_sample(frames, fx, seed)
    clip_s = _extrapolate(t_unet, frames, fx)
    cores = _CPU_WEIGHTS["cores"]
    return {"value": round(FRAMES / clip_s, 6), "unit": "frames/s", "cores": cores, "kind": "port",
            "sample": f"1 CFG UNet3D forward on {frames} of {FRAMES} frames at 64x64 latents ({t_unet:.1f} s) + reference "
                      f"UNet ({fx['t_ref']:.1f} s) + 1 VAE decode frame ({fx['t_dec']:.1f} s) + 1 VAE encode frame "
                      f"({fx['t_enc']:.1f} s), fp32, {cores} threads; clip = {DDIM_STEPS} x forward x {FRAMES}/{frames} + "
                      f"{FRAMES} decodes + 2 encodes + reference UNet",
            "extrapolated_clip_seconds": round(clip_s, 1)}


def run_reference(args):
    """`--impl reference`: the oracle port on the host cores, `warmup` + `steps` bounded samples (see module docstring).
    The whole run is sized to ~4 minutes: f_s frames per sample follow from a one-frame probe."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    t_run = time.perf_counter()
    budget_s = 240.0
    fx = cpu_fixed_parts(0)
    probe = cpu_unet_sample(1, fx, 0)
    n = args.warmup + args.steps
    left = budget_s - (time.perf_counter() - t_run)
    f_s = int(max(1, min(FRAMES, (left / n) / max(probe, 1e-3))))
    while FRAMES % f_s:  # a divisor of 24 keeps the extrapolation factor integral
        f_s -= 1
    walls, vals = [], []
    for i in range(n):
        t = cpu_unet_sample(f_s, fx, i)
        if i >= args.warmup:
            walls.append(t)
            vals.append(FRAMES / _extrapolate(t, f_s, fx))
    v = statistics.mean(vals)
    cores = _CPU_WEIGHTS["cores"]
    cpu = {"value": round(v, 6), "unit": "frames/s", "cores": cores, "kind": "port",
           "sample": f"per step: 1 CFG UNet3D forward on {f_s} of {FRAMES} frames at 64x64 latents (mean "
                     f"{statistics.mean(walls):.2f} s); once: reference UNet {fx['t_ref']:.1f} s, VAE decode frame "
                     f"{fx['t_dec']:.1f} s, VAE encode frame {fx['t_enc']:.1f} s; fp32, {cores} threads; clip = "
                     f"{DDIM_STEPS} x forward x {FRAMES}/{f_s} + {FRAMES} decodes + 2 encodes + reference UNet",
           "extrapolated_clip_seconds": round(FRAMES / v, 1), "frames_per_sample": f_s}
    line = {"impl": "reference", "metric": METRIC, "value": round(v, 6), "unit": "frames/s",
            "n_gpus": int(os.environ.get("WORLD_SIZE", 1)), "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(1e3 * statistics.mean(walls), 1), "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": dict(CONFIG),
            "note": "value = clip-extrapolated frames/s of the bounded per-step sample; ms_per_step = wall time of a "
                    "sample step (see cpu_baseline.sample)",
            "cpu_baseline": cpu,
            "e2e": {"value": round(v, 6), "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, help="BASELINE.json config number: 2 (default, the metric), 4, 5")
    ap.add_argument("--dump-calls", default=None, help="write every profiled C-ABI call (name, flops, bytes, ms) as CSV")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write what the last timed step returned (latents, videos) as DIR/<name>.npy, float32")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU sample (development runs)")
    ap.add_argument("--no-breakdown", action="store_true",
                    help="skip the two extra diagnostic clips (event-bracketed calls, CUPTI table): roofline = null")
    ap.add_argument("--one-clip", action="store_true",
                    help="run exactly one device-resident clip and exit (for `ncu` launch lists; not a bench value)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.one_clip or args.impl == "reference"):
        ap.error("--dump-outputs writes the timed steps of our engine: not with --one-clip or --impl reference")
    select_config(args.config)
    if args.impl == "reference":
        run_reference(args)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device. The engine has no CPU fallback (use --impl reference for the CPU port).")
    args.warmup = max(args.warmup, 3)
    run_ours(args)


if __name__ == "__main__":
    main()
