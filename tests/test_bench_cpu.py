"""bench.py's host-side contract, without a GPU and without minutes of CPU work: the synthetic inputs are seeded, the
BASELINE configurations select what they say, and the reference arm (`--impl reference`) prints the line the driver
parses - with the oracle's timed pieces replaced by a stub clock, so that only bench.py's own logic runs here (the real
arm takes ~4 minutes of host time; it was run as is: 0.0095 frames/s on the 8-thread build container)."""
import argparse
import json

import numpy as np
import pytest


@pytest.fixture()
def bench_mod():
    import importlib

    import bench
    yield bench
    importlib.reload(bench)  # select_config() mutates module globals


def test_synthetic_inputs_are_seeded_and_shaped(bench_mod):
    b = bench_mod
    r1, p1, k1 = b.synthetic_inputs(3, 64, seed=0)
    r2, p2, k2 = b.synthetic_inputs(3, 64, seed=0)
    assert r1.size == (64, 64) and r1.mode == "RGB" and len(p1) == len(k1) == 3
    assert r1.tobytes() == r2.tobytes() and all(a.tobytes() == c.tobytes() for a, c in zip(p1, p2))
    assert all(np.asarray(k).min() == 255 for k in k1)                      # animate mode: white backgrounds (init_bk)
    assert all(0 < (np.asarray(p) > 10).sum() < 64 * 64 * 3 for p in p1)    # a coloured blob on black
    _, _, kn = b.synthetic_inputs(3, 64, seed=0, noise_bk=True)
    assert len({k.tobytes() for k in kn}) == 3                              # edit mode: a distinct background per frame


def test_select_config_matches_baseline_json(bench_mod):
    b = bench_mod
    configs = json.loads((b.ROOT / "BASELINE.json").read_text())["configs"]
    assert "512" in configs[1] and "24-frame" in configs[1] and "20 DDIM" in configs[1]
    assert (b.WIDTH, b.FRAMES, b.DDIM_STEPS, b.DTYPE_NAME) == (512, 24, 20, "fp16")
    b.select_config(4)
    assert "768" in configs[3] and "48-frame" in configs[3] and "30 DDIM" in configs[3] and "bf16" in configs[3]
    assert (b.WIDTH, b.HEIGHT, b.FRAMES, b.DDIM_STEPS, b.DTYPE_NAME) == (768, 768, 48, 30, "bf16")
    assert b.METRIC == "frames/sec @ 768x768x48f, 30 DDIM steps" and b.CONFIG["frames"] == 48
    with pytest.raises(SystemExit):
        b.select_config(7)


def test_select_config_5_is_the_edit_clip(bench_mod):
    b = bench_mod
    b.select_config(5)
    assert (b.WIDTH, b.FRAMES, b.DDIM_STEPS, b.DTYPE_NAME, b.NOISE_BK) == (512, 64, 20, "fp16", True)


def test_reference_arm_line_and_sample_sizing(bench_mod, monkeypatch, capsys):
    """run_reference(): warm-up + steps samples of f_s frames, f_s a divisor of 24 sized from a one-frame probe to a
    ~4 minute budget; the printed line carries the keys the driver reads, `value` = clip-extrapolated frames/s,
    `ms_per_step` = the real wall time of a sample."""
    b = bench_mod
    per_frame, calls = 2.0, []
    monkeypatch.setattr(b, "cpu_fixed_parts", lambda seed=0: {"t_ref": 3.0, "t_dec": 5.0, "t_enc": 2.0, "banks": None, "ehs": None})

    def fake_sample(frames, fixed, seed=0):
        calls.append(frames)
        return per_frame * frames
    monkeypatch.setattr(b, "cpu_unet_sample", fake_sample)
    b._CPU_WEIGHTS["cores"] = 4
    monkeypatch.delenv("RANK", raising=False)
    b.run_reference(argparse.Namespace(steps=3, warmup=1))
    line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert calls[0] == 1 and len(calls) == 1 + 4          # the probe, then warm-up + steps samples
    f_s = calls[1]
    assert 24 % f_s == 0 and all(c == f_s for c in calls[1:])
    assert f_s == 24                                      # 240 s / 4 samples / 2 s per frame = 30 frames -> capped at the clip
    clip_s = 20 * (per_frame * f_s) * (24 / f_s) + 24 * 5.0 + 2 * 2.0 + 3.0
    assert line["impl"] == "reference" and line["metric"] == b.METRIC and line["unit"] == "frames/s"
    assert line["value"] == pytest.approx(24 / clip_s, rel=1e-4) and line["higher_is_better"] is True
    assert line["ms_per_step"] == pytest.approx(1e3 * per_frame * f_s) and line["steps"] == 3 and line["warmup"] == 1
    assert line["e2e"] == {"value": line["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] == 4 and cb["value"] == line["value"] and "24 frames" in cb["sample"]
    assert line["config"] == b.CONFIG

    # a slow host: the sample shrinks to what fits the budget, still a divisor of 24
    calls.clear()
    per_frame = 9.0
    b.run_reference(argparse.Namespace(steps=5, warmup=3))
    capsys.readouterr()
    assert calls[1] == 3 and 24 % calls[1] == 0           # 240 / 8 / 9 = 3.3 frames

    # the other ranks of a torchrun launch exit without work
    calls.clear()
    monkeypatch.setenv("RANK", "1")
    b.run_reference(argparse.Namespace(steps=1, warmup=0))
    assert calls == [] and capsys.readouterr().out == ""


def test_usable_cores_and_extrapolation(bench_mod):
    b = bench_mod
    assert 1 <= b.usable_cores() <= 4096
    fx = {"t_ref": 1.0, "t_dec": 2.0, "t_enc": 3.0}
    assert b._extrapolate(10.0, 8, fx) == 20 * 10.0 * 3 + 24 * 2.0 + 2 * 3.0 + 1.0


def test_dump_outputs_budget_and_sample(bench_mod, tmp_path):
    """--dump-outputs: small outputs whole, a large one as a fixed seeded sample; float32, DUMP_BYTES in all."""
    import torch
    b = bench_mod
    lat = torch.randn(1, 4, 24, 64, 64, dtype=torch.float16)
    vid = torch.rand(1, 3, 24, 512, 512, dtype=torch.float16)
    for d in ("a", "b"):
        b.dump_outputs({"latents": lat, "videos": vid}, tmp_path / d)
    got = {n: np.load(tmp_path / "a" / f"{n}.npy") for n in ("latents", "videos")}
    assert got["latents"].dtype == got["videos"].dtype == np.float32
    assert np.array_equal(got["latents"], lat.float().numpy())
    assert got["videos"].ndim == 1 and 0 < got["videos"].size < vid.numel()
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) < 64 * 1000 * 1000
    assert np.array_equal(got["videos"], np.load(tmp_path / "b" / "videos.npy"))
    assert np.isin(got["videos"], vid.float().numpy().reshape(-1)).all()
