"""CPU: the parts of bench.py's contract that do not need a GPU — both arms describe the same workload, the synthetic
inputs have BASELINE.json's configs[2] shapes, the clock sampler and peak lookup degrade gracefully."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def test_config_is_shared_by_both_arms_and_names_the_workload():
    cfg = bench.bench_config(3)
    assert cfg == bench.bench_config(3)
    assert "SDXL 1024x1024" in cfg["workload"] and "5 region prompts" in cfg["workload"]
    assert cfg["passes_per_step"] == 8 == bench.passes_per_step(bench.CONFIGS[3])
    assert abs(cfg["unet_tflop_per_step"] - 8 * 6.7612) < 1e-6
    assert "L2" in cfg["l2"]
    json.dumps(cfg)
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert "steps/sec" in base["metric"] or "steps/s" in base["metric"]
    # one bench configuration per BASELINE.json config, pass counts as SURVEY 8d states them
    assert len(bench.CONFIGS) == len(base["configs"]) == 5
    assert [bench.passes_per_step(bench.CONFIGS[i]) for i in range(1, 6)] == [2, 6, 8, 11, 13]
    assert bench.bench_config(5)["passes_per_step"] == 4 * 13


def test_timed_steps_cover_both_injection_regimes():
    """The K timed schedule positions are spread over the schedule; with inject_selfattn=0.5 about half of them fall in
    each regime, so the timed region cannot sit entirely on one side of the step-20 flip (round-1 defect)."""
    from rtti_b200.schedulers import EulerDiscreteScheduler
    sch = EulerDiscreteScheduler()
    sch.set_timesteps(41)
    for k in (6, 20):
        idx = bench.spread(k, 41)
        assert len(idx) == k and idx == sorted(idx) and 0 <= idx[0] and idx[-1] <= 40
        on = sum(1 for i in idx if float(sch.timesteps[i]) > 500.0)
        assert abs(on - k / 2) <= 1


def test_image_groups_for_the_batched_config():
    assert bench.image_groups(1, 0, 4) == ([0, 1, 2, 3], 1)
    assert bench.image_groups(2, 1, 4) == ([2, 3], 1)
    assert bench.image_groups(4, 3, 4) == ([3], 1)
    assert [bench.image_groups(8, r, 4) for r in range(8)] == [([r // 2], 2) for r in range(8)]


def test_synthetic_workload_shapes():
    wl = bench.synth_workload(bench.CONFIGS[3])
    n = bench.CONFIGS[3]["regions"]
    assert wl["ctx"].shape == (n + 1, 77, 2048) and wl["pooled"].shape == (n + 1, 1280)
    assert wl["latents"].shape == (1, 4, 128, 128)
    assert len(wl["masks"]) == n and all(m.shape == (1, 4, 128, 128) for m in wl["masks"])
    tot = sum(m for m in wl["masks"])
    assert float((tot - 1).abs().max()) < 1e-5                      # region masks partition the latent
    assert wl["tfd"]["color_obj_atten"][0].shape == (1, 4, 1024, 1024)
    assert wl["tfd"]["target_RGB"][0].shape == (1, 3, 1, 1)
    sd = bench.synth_workload(bench.CONFIGS[2])
    assert sd["ctx"].shape == (4, 77, 768) and sd["latents"].shape == (1, 4, 64, 64) and "target_RGB" not in sd["tfd"]


def test_clock_sampler_and_peaks_degrade_gracefully():
    s = bench.ClockSampler(0)          # no nvidia-smi in the CPU container: must not raise
    out = s.stop()
    assert set(out) >= {"sm_mhz", "sm_max_mhz", "reasons"}
    hbm, burst, sust, src = bench.peaks()
    assert hbm > 1000 and burst >= sust > 100 and src in ("measured", "fallback")
    assert bench.host_threads() >= 1


def test_reference_arm_other_ranks_exit_quietly():
    """Under torchrun (N > 1) rank 0 alone prints the reference line; the other ranks exit 0 without work."""
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=120, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_dump_outputs_writes_float32_npy(tmp_path):
    import numpy as np
    import torch
    lat = torch.randn(1, 4, 8, 8).half()
    bench.dump_outputs(str(tmp_path / "out"), {"latents": lat, "color_loss": torch.tensor([0.25])})
    got = np.load(tmp_path / "out" / "latents.npy")
    assert got.dtype == np.float32 and np.array_equal(got, lat.float().numpy())
    assert np.load(tmp_path / "out" / "color_loss.npy").tolist() == [0.25]


def test_steps_must_be_positive():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 2 and "--steps" in r.stderr


def test_committed_bench_lines_carry_every_contract_key():
    """The JSON lines measured on the B200 boxes this round (profiles/r02_bench_*.json) against the keys the driver's
    contract lists: metric / value / unit / n_gpus / steps / warmup / ms_per_step / higher_is_better / scaling /
    vs_baseline / dtype / data / config.workload / clocks / gpu_launches / e2e{value, unit, h2d, d2h}; config 3 at N = 1
    also roofline{bound, achieved, peak, unit, frac, traffic}; N > 1 lines the rank-identity flag."""
    import glob
    paths = sorted(glob.glob(os.path.join(ROOT, "profiles", "r02_bench_n*_config*.json")))
    assert len(paths) >= 8
    for p in paths:
        line = [l for l in open(p) if l.startswith("{")][-1]
        d = json.loads(line)
        for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                  "vs_baseline", "dtype", "data", "config", "clocks", "gpu_launches", "e2e"):
            assert k in d, (p, k)
        assert d["metric"] == "denoising steps/sec" and d["unit"] == "steps/s" and d["higher_is_better"] is True
        assert d["scaling"] == "strong" and d["vs_baseline"] is None and d["data"] == "synthetic" and d["warmup"] >= 3
        assert "workload" in d["config"] and "model" not in d["config"]
        assert abs(d["value"] - d["steps"] / (d["ms_per_step"] * d["steps"] * 1e-3)) < 1e-6 * d["value"]
        assert d["gpu_launches"] > 0
        e = d["e2e"]
        assert e["value"] > 0 and e["unit"] == "steps/s" and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0
        assert not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
        if d["config"]["config_id"] == 3:
            r = d["roofline"]
            assert r["bound"] == "tensor" and r["unit"] == "TFLOP/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
            assert r["traffic"] and (0.3 < r["frac"] < 0.7 if d["n_gpus"] == 1 else 0.05 < r["frac"] < 0.7)   # batch-1 passes at N = 8
            assert d["roofline_cross_attention"]["bound"] == "hbm"
        if d["n_gpus"] > 1:
            assert d["ranks_bit_identical"] is True
            if d.get("single_gpu_check"):
                assert d["single_gpu_check"]["pass"] is True
