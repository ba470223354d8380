"""bench.py — denoising steps/sec of the region-diffusion hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--config C]        # product arm (one rank per GPU under torchrun)
    python bench.py --impl reference --steps K --warmup W [--config C] # reference arm: CPU oracle port on the host cores

`--config` selects one of BASELINE.json's five workloads (SURVEY §8d); the default, 3, is the one the metric is
quoted on: SDXL 1024^2, 5 region prompts, color_guidance_weight=1, inject_selfattn=0.5, inject_background=0.5 ->
8 UNet passes per step (uncond, base + font sizes, reference uncond / base, 4 regions) run as one batched call,
region blend + CFG + Euler, colour guidance through the fp32 SDXL VAE decoder. One "step" = one iteration of
models/region_diffusion_sdxl.py:779-878 (SD1.5: models/region_diffusion.py:99-173). Random weights of the real
architectures, seeded synthetic inputs (no checkpoints / datasets in this environment).

The K timed steps are taken at schedule positions spread evenly over the sampling schedule, so that the two regimes
of a run (self-attention injection on for t > (1 - inject_selfattn) * 1000, off afterwards) are timed in the proportion
a full sampling run has them. Every CUDA-graph / exchange / cuDNN-autotune state the timed steps can reach is
executed once before the timed region.

`--dump-outputs DIR` writes what the last timed step returned (latents; SDXL configs also the guided noise prediction
and the colour loss) as DIR/<name>.npy in float32. Weights and inputs are seeded, so two builds run with the same
arguments can be compared output for output.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GUIDANCE = 8.5
UNET_PASS_GFLOP = {"sdxl": 6761.2, "sd15": 803.3}  # SURVEY §8d [probe], batch-1 UNet forward

CONFIGS = {
    1: dict(model="sd15", regions=1, schedule=10, inject_selfattn=0.0, inject_background=0.0, color=False, images=1,
            name="SD1.5 512x512 plain-text single prompt, 10 steps, 1 region (BASELINE configs[0])"),
    2: dict(model="sd15", regions=3, schedule=41, inject_selfattn=0.3, inject_background=0.5, color=False, images=1,
            name="SD1.5 512x512 footnote example shape: 3 regions, 41 steps, token-map capture pass + rich pass (configs[1])"),
    3: dict(model="sdxl", regions=5, schedule=41, inject_selfattn=0.5, inject_background=0.5, color=True, images=1,
            name="SDXL 1024x1024 font-color example shape: 5 region prompts, color_guidance_weight=1, inject_selfattn=0.5, "
                 "inject_background=0.5, 41-step Euler schedule (configs[2])"),
    4: dict(model="sdxl", regions=8, schedule=41, inject_selfattn=0.0, inject_background=0.4, color=False, images=1,
            name="SDXL 1024x1024 font-style example shape: 8 region prompts, inject_background=0.4, 41 steps (configs[3])"),
    5: dict(model="sdxl", regions=10, schedule=50, inject_selfattn=0.5, inject_background=0.5, color=False, images=4,
            name="SDXL 1024x1024 batch of 4 images x 10 region prompts, inject_selfattn=0.5, inject_background=0.5, 50 steps "
                 "(configs[4]); one step = one denoising iteration of all 4 images"),
}


def passes_per_step(cfg):
    inj = cfg["inject_selfattn"] > 0 or cfg["inject_background"] > 0
    return 2 + (2 if inj else 0) + (cfg["regions"] - 1)


def bench_config(cfg_id):
    """`config` of the JSON line: identical for the product arm and the --impl reference arm."""
    cfg = CONFIGS[cfg_id]
    pps = passes_per_step(cfg)
    d = {"workload": cfg["name"], "config_id": cfg_id, "passes_per_step": pps * cfg["images"],
         "unet_tflop_per_step": pps * cfg["images"] * UNET_PASS_GFLOP[cfg["model"]] / 1e3,
         "timed_steps": "schedule positions spread evenly over the sampling schedule (both injection regimes)",
         "l2": "inputs larger than L2: the fp16 UNet weights (5.1 GB SDXL / 1.7 GB SD1.5) stream every step"}
    if cfg["color"]:
        d["vae"] = "SDXL AutoencoderKL decoder, random weights, fp32/TF32, fwd+bwd inside the step"
    return d


def spread(k, n):
    """k schedule positions spread evenly over an n-step schedule."""
    return [min(n - 1, int((i + 0.5) * n / k)) for i in range(k)]


def synth_workload(cfg, image=0):
    import torch
    g = torch.Generator().manual_seed(7 + 101 * image)
    N = cfg["regions"]
    xl = cfg["model"] == "sdxl"
    h = w = 128 if xl else 64
    ctx = torch.randn(N + 1, 77, 2048 if xl else 768, generator=g)
    pooled = torch.randn(N + 1, 1280, generator=g)
    latents = torch.randn(1, 4, h, w, generator=g)
    logits = torch.randn(N, 1, 8, 8, generator=g)
    up = torch.nn.functional.interpolate(logits, (h, w), mode="bicubic", align_corners=False)
    m = torch.softmax(up * 3.0, dim=0)
    masks = [m[i:i + 1].repeat(1, 4, 1, 1) for i in range(N)]
    tfd = {"word_pos": torch.LongTensor([2, 5, 9]), "font_size": torch.FloatTensor([2.0, 0.5, -1.5])}
    if cfg["color"]:
        color_mask = torch.nn.functional.interpolate(masks[0], (h * 8, w * 8), mode="bicubic", antialias=True).clamp(0, 1)
        tfd.update({"target_RGB": [torch.tensor([253, 108, 158.0]).reshape(1, 3, 1, 1) / 255.0], "guidance_start_step": 999,
                    "color_guidance_weight": 1.0, "color_obj_atten": [color_mask], "color_obj_atten_all": masks[0].clone()})
    return dict(ctx=ctx, pooled=pooled, latents=latents, masks=masks, tfd=tfd)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                       "-i", str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 8:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if sm:
            sm.sort()
            out = {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        return out


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops", 1590.0), d.get("bf16_tflops_sustained", 1400.0), "measured"
    return 6650.0, 1590.0, 1400.0, "fallback"


def ncu_traffic(kernel_key):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` capture of this
    round (profiles/r02_ncu_traffic.json, written from the .ncu-rep by tools/ncu_traffic.py), or None."""
    p = os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")
    if not os.path.exists(p):
        return None, None
    with open(p) as f:
        d = json.load(f)
    e = d.get(kernel_key)
    return (e["bytes_per_launch"], e["note"]) if e else (None, None)


def dump_outputs(out_dir, arrays):
    """--dump-outputs: every tensor of `arrays` as out_dir/<name>.npy, float32."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


def host_threads():
    """CPU threads this process may really use: affinity mask capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(math.ceil(int(quota) / int(period)))))
    except Exception:
        pass
    return n


# ------------------------------------------------------------------------------------------- CPU oracle (reference arm)
def oracle_unet(model):
    """(state dict, config, inputs) of the CPU fp32 oracle UNet, torch-random weights (N(0, 1/fan_in))."""
    import torch
    from oracle import unet_oracle as uo
    torch.set_num_threads(host_threads())
    cfg = uo.sdxl_config() if model == "sdxl" else uo.sd15_config()
    g = torch.Generator().manual_seed(0)
    sd = {}
    for k, shp in uo.param_shapes(cfg).items():
        if len(shp) >= 2:
            sd[k] = torch.empty(shp).normal_(generator=g).div_(math.sqrt(float(torch.Size(shp[1:]).numel())))
        else:
            sd[k] = torch.ones(shp) if k.endswith("weight") else torch.zeros(shp)
    xl = model == "sdxl"
    s = 128 if xl else 64
    x = torch.randn(1, 4, s, s, generator=g)
    ctx = torch.randn(1, 77, 2048 if xl else 768, generator=g)
    added = {"text_embeds": torch.randn(1, 1280, generator=g),
             "time_ids": torch.tensor([[1024.0, 1024, 0, 0, 1024, 1024]])} if xl else None
    return sd, cfg, x, ctx, added


def cpu_oracle_pass_times(model, n_samples, warm):
    """Wall seconds of `n_samples` WHOLE batch-1 UNet passes of the CPU oracle (fp32, all usable host threads)."""
    import torch
    from oracle import unet_oracle as uo
    sd, cfg, x, ctx, added = oracle_unet(model)
    times = []
    with torch.no_grad():
        for i in range(warm + n_samples):
            t0 = time.perf_counter()
            uo.unet_forward(sd, cfg, x, torch.tensor(981.0), ctx, added)
            dt = time.perf_counter() - t0
            if i >= warm:
                times.append(dt)
    return times, torch.get_num_threads()


def cpu_oracle_guidance_time():
    """Wall seconds of ONE colour-guidance evaluation of the CPU oracle at 1024^2: fp32 VAE decode, clamp, masked-mean
    MSE, backward to the latents INCLUDING the weight gradients the reference computes and discards (sdxl.py:856-865)."""
    import torch
    from oracle import sampler_oracle as sam, vae_oracle as vo
    torch.set_num_threads(host_threads())
    cfg = vo.VAEConfig()
    sd = vo.make_state_dict(cfg, 1)
    for v in sd.values():
        v.requires_grad_(True)
    wl = synth_workload(CONFIGS[3])
    g = torch.Generator().manual_seed(3)
    lat = torch.randn(1, 4, 128, 128, generator=g)
    eps = torch.randn(1, 4, 128, 128, generator=g)
    alphas = torch.linspace(0.999, 0.01, 1000)
    t0 = time.perf_counter()
    sam.color_guidance(lat, eps, 500, alphas, lambda z: vo.decode(sd, cfg, z), cfg.scaling_factor, wl["tfd"], xl=True)
    return time.perf_counter() - t0


def run_reference(args, rank):
    """Reference arm: the reference's own algorithm on the host cores. The reference is pure Python on top of
    `diffusers`, which is not installed and cannot be on the GPU box, so this is the CPU oracle port (oracle/, pinned
    against the unmodified reference by tests/golden): kind "port". Each timed "step" is a bounded sample of the
    workload: ONE WHOLE batch-1 UNet pass (a step consists of `passes_per_step` of them); the colour guidance of a step
    (config 3) is evaluated once, whole, outside the K samples. Nothing is extrapolated by FLOPs:
        seconds per step = passes_per_step x mean(seconds per whole pass) + seconds per whole guidance evaluation."""
    if rank != 0:
        return
    cfg = CONFIGS[args.config]
    pps = passes_per_step(cfg) * cfg["images"]
    times, threads = cpu_oracle_pass_times(cfg["model"], args.steps, min(args.warmup, 1))
    t_pass = sum(times) / len(times)
    t_guid = cpu_oracle_guidance_time() if cfg["color"] else 0.0
    t_step = pps * t_pass + t_guid
    v = 1.0 / t_step
    sample = (f"{len(times)} timed samples, each ONE WHOLE batch-1 {cfg['model']} UNet pass of the fp32 CPU oracle "
              f"(mean {t_pass:.2f} s, min {min(times):.2f}, max {max(times):.2f}); one step = {pps} such passes"
              + (f" + one whole colour-guidance evaluation (fp32 VAE decode + backward incl. weight gradients, measured once: "
                 f"{t_guid:.1f} s)" if cfg["color"] else "")
              + f" = {t_step:.1f} s/step; blend/CFG/scheduler (<0.1 %) not included; no FLOP extrapolation")
    print(json.dumps({
        "impl": "reference", "metric": "denoising steps/sec", "value": v, "unit": "steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": min(args.warmup, 1),
        "ms_per_step": 1000.0 * t_pass, "ms_per_step_note": "wall time of one timed sample (one whole UNet pass), so that "
        "steps x ms_per_step is the timed region of this run; the full-step time is seconds_per_full_step",
        "seconds_per_full_step": t_step, "seconds_per_pass": t_pass, "seconds_per_guidance": t_guid,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": bench_config(args.config),
        "cpu_baseline": {"value": v, "unit": "steps/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


# ------------------------------------------------------------------------------------------- product arm, SDXL configs
def solo_check(model, fresh_state, workload, st_par, idx, dist, rank, world):
    """--check: every rank repeats the same step sequence as a single-GPU run (all passes local, no exchange, no stripes)
    and compares its latents with the region-parallel result: stated tolerance 0.5 % of the dynamic range + 3 %."""
    import torch
    solo = [dist.new_group([r]) for r in range(world)][rank]
    saved = (model.region_group, model.fused_exchange, model.stripe_guidance)
    model.region_group, model.stripe_guidance = solo, False
    st = fresh_state(workload)
    with torch.no_grad():
        for i in idx:
            model.rich_text_step(st, i)
    torch.cuda.synchronize()
    model.region_group, model.fused_exchange, model.stripe_guidance = saved
    a, b = st_par.latents.float(), st.latents.float()
    err = (a - b).abs()
    tol = 5e-3 * float(b.abs().max()) + 3e-2 * b.abs()
    res = {"max_err": float(err.max()), "mean_err": float(err.mean()), "ref_absmax": float(b.abs().max()),
           "frac_outside_tolerance": float((err > tol).float().mean()), "steps_compared": len(idx)}
    t = torch.tensor([res["frac_outside_tolerance"], res["max_err"]], device=a.device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    res["frac_outside_tolerance"], res["max_err"] = float(t[0]), float(t[1])
    res["pass"] = res["frac_outside_tolerance"] == 0.0
    return res


def image_groups(world, rank, n_images):
    """Config 5: data-parallel over images first, region-parallel inside. Returns (images of this rank, ranks per image).
    world >= images: world // images ranks work on one image; else every rank owns images // world whole images."""
    if world >= n_images:
        rpi = world // n_images
        return [min(rank // rpi, n_images - 1)], rpi
    per = n_images // world
    return list(range(rank * per, (rank + 1) * per)), 1


def run_product_xl(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from rtti_b200 import ops
    from rtti_b200.region_diffusion_sdxl import RegionDiffusionXL
    cfg = CONFIGS[args.config]
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    model = RegionDiffusionXL.from_synthetic(seed=0, device=dev, with_vae=cfg["color"])
    n_t = cfg["schedule"]
    model.scheduler.set_timesteps(n_t)
    timesteps = model.scheduler.timesteps
    time_ids = torch.tensor([[1024.0, 1024, 0, 0, 1024, 1024]], device=dev)
    my_images = [0]
    if cfg["images"] > 1:
        my_images, rpi = image_groups(world, rank, cfg["images"])
        if world > 1:   # every rank creates every group, in the same order; region-parallel sharding stays inside a group
            for g0 in range(0, world, rpi):
                ranks = list(range(g0, min(world, g0 + rpi)))
                grp = dist.new_group(ranks)
                if rank in ranks:
                    model.region_group = grp
    workloads = [synth_workload(cfg, im) for im in my_images]

    def fresh_state(src):
        tfd = dict(src["tfd"])
        for key in ("color_obj_atten", "target_RGB"):
            if key in tfd:
                tfd[key] = [m.to(dev, non_blocking=True) for m in tfd[key]]
        if "color_obj_atten_all" in tfd:
            tfd["color_obj_atten_all"] = tfd["color_obj_atten_all"].to(dev, non_blocking=True)
        lat = src["latents"].to(dev, torch.float16, non_blocking=True) * model.scheduler.init_noise_sigma
        model.masks = [m.to(dev, non_blocking=True) for m in src["masks"]]
        return model.prepare_rich_text(src["ctx"].to(dev, torch.float16, non_blocking=True),
                                       src["pooled"].to(dev, torch.float16, non_blocking=True), time_ids, lat, timesteps,
                                       GUIDANCE, cfg["color"], cfg["inject_selfattn"], cfg["inject_background"], tfd)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    states = [fresh_state(w) for w in workloads]
    # every state a timed step can be in: injection on (i = 0), the background-injection blend step, injection off (last)
    warm_idx = sorted({0, min(n_t - 1, int(cfg["inject_background"] * n_t)), n_t - 1})
    w_idx = spread(args.warmup, n_t)
    t_idx = spread(args.steps, n_t)
    def peer_errors():
        """True on every rank if any rank's peer-memory waits (RemoteQK, exchange, stripe arena) timed out."""
        bad = any(rq is not None and rq.error() for rq in model._remote.values())
        for obj in list(model._exchanges.values()) + [e.arena for e in model._stripe_engines.values()]:
            try:
                obj.check()
            except RuntimeError:
                bad = True
        t = torch.tensor([1.0 if bad else 0.0], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return bool(t.item() > 0)

    fallback = None
    with torch.no_grad():
        for i in warm_idx + w_idx:
            for st in states:
                model.rich_text_step(st, i)
        barrier()
        if world > 1 and peer_errors():
            # safety net: a peer wait timed out during warm-up (never seen; the kernels give up after seconds instead of
            # hanging). Fall back to the round-1 scheme — pass D replicated, eager guidance — and say so in the line.
            fallback = "peer wait timed out in warm-up: remote_qk and graph_guidance disabled for this run"
            print("bench.py: " + fallback, file=sys.stderr, flush=True)
            model.remote_qk = model.graph_guidance = False
            states = [fresh_state(w) for w in workloads]
            for i in warm_idx + w_idx:
                for st in states:
                    model.rich_text_step(st, i)
            barrier()
        # ------------------------------------------------------------- device-resident timing
        clocks = ClockSampler(local_rank) if rank == 0 else None
        launches0 = ops.LAUNCHES
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.cuda.nvtx.range_push("timed")
        for i in t_idx:
            for st in states:
                model.rich_text_step(st, i)
        torch.cuda.nvtx.range_pop()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        launches = ops.LAUNCHES - launches0
        clk = clocks.stop() if clocks else None
    if args.dump_outputs:   # the last timed step's result, written once per image by the lowest rank that holds it
        out = {}
        for im, st in zip(my_images, states):
            holders = [r for r in range(world) if cfg["images"] == 1 or im in image_groups(world, r, cfg["images"])[0]]
            if rank == holders[0]:
                pre = f"image{im}_" if cfg["images"] > 1 else ""
                out[pre + "latents"], out[pre + "noise_pred"] = st.latents, st.noise_pred
        if rank == 0 and "color_loss" in model.last_step_stats:
            out["color_loss"] = model.last_step_stats["color_loss"]
        dump_outputs(args.dump_outputs, out)
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    for st in states:
        assert bool(torch.isfinite(st.latents.float()).all()), "non-finite latents"
    # the blend / scheduler / guidance are replicated deterministically: all ranks of a region-parallel group must hold
    # bit-identical latents after the timed loop (checked on every run; --check adds the single-GPU comparison)
    ranks_identical = None
    if world > 1:
        h = torch.stack([st.latents.view(torch.int16).to(torch.int64).sum() for st in states]).reshape(1, -1)
        hs = [torch.empty_like(h) for _ in range(world)]
        dist.all_gather(hs, h)
        grp = range(world) if cfg["images"] == 1 else [r for r in range(world) if image_groups(world, r, cfg["images"])[0] == my_images]
        ranks_identical = all(bool(torch.equal(hs[r], h)) for r in grp)
        assert ranks_identical, "latents differ between the ranks of a region-parallel group"
    check = None
    if args.check and world > 1 and cfg["images"] == 1:
        check = solo_check(model, fresh_state, workloads[0], states[0], warm_idx + w_idx + t_idx, dist, rank, world)

    # ------------------------------------------------------------- end to end: host buffers every step
    def pin(w):
        p = {k: (v.pin_memory() if torch.is_tensor(v) else v) for k, v in w.items()}
        p["masks"] = [m.pin_memory() for m in w["masks"]]
        p["tfd"] = dict(w["tfd"])
        if "color_obj_atten" in w["tfd"]:
            p["tfd"]["color_obj_atten"] = [m.pin_memory() for m in w["tfd"]["color_obj_atten"]]
            p["tfd"]["color_obj_atten_all"] = w["tfd"]["color_obj_atten_all"].pin_memory()
        return p

    pinned = [pin(w) for w in workloads]
    h2d = 0
    for p in pinned:
        ts = [p["ctx"], p["pooled"], p["latents"], *p["masks"]]
        if "color_obj_atten" in p["tfd"]:
            ts += [*p["tfd"]["color_obj_atten"], p["tfd"]["color_obj_atten_all"]]
        h2d += sum(x.numel() * x.element_size() for x in ts)
    # Results are read back through pinned double buffers, ONE STEP DEEP: step k's latents / loss are copied to the host
    # asynchronously right after its launches and consumed (event wait + host read) after step k+1 has been issued, so the
    # host work of a step (input staging, launches) overlaps the device work of the previous one. Every step still pays
    # its own H2D of all inputs and its own D2H of the result inside the timed region.
    host_lat = [torch.empty(1, 4, 128, 128, dtype=torch.float16).pin_memory() for _ in range(2)]
    host_loss = [torch.zeros(1, dtype=torch.float32).pin_memory() for _ in range(2)]
    loss = None

    def drain(pend):
        ev, slot = pend
        ev.synchronize()
        assert bool(torch.isfinite(host_lat[slot][0, 0, 0, :8].float()).all())
        return float(host_loss[slot][0]) if cfg["color"] else None

    with torch.no_grad():
        barrier()
        t0 = time.perf_counter()
        pending, k = None, 0
        for i in t_idx:
            for st, p in zip(states, pinned):
                s2 = fresh_state(p)                      # H2D of this step's inputs from pinned host memory
                s2.kv_caches = st.kv_caches              # prompt K/V projections and the captured UNet graphs are
                s2.graphs = st.graphs                    # per-prompt state, kept across steps
                model.rich_text_step(s2, i)              # the public step call
                host_lat[k & 1].copy_(s2.latents, non_blocking=True)       # D2H of the step result (async, pinned)
                if cfg["color"] and "color_loss" in model.last_step_stats:
                    host_loss[k & 1].copy_(model.last_step_stats["color_loss"], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record()
                if pending is not None:
                    loss = drain(pending)
                pending, k = (ev, k & 1), k + 1
        loss = drain(pending)
        barrier()
        e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_s = float(te.item())
    d2h = (host_lat[0].numel() * 2 + (4 if cfg["color"] else 0)) * len(states)

    # ------------------------------------------------------------- whole sampling loop, wall clock (graphs warm)
    with torch.no_grad():
        barrier()
        t0 = time.perf_counter()
        for st, p in zip(states, pinned):
            s2 = fresh_state(p)
            s2.kv_caches, s2.graphs = st.kv_caches, st.graphs
            for i in range(n_t):
                model.rich_text_step(s2, i)
            host_lat[0].copy_(s2.latents, non_blocking=False)
        barrier()
        loop_s = time.perf_counter() - t0
    tl = torch.tensor([loop_s], device=dev)
    if world > 1:
        dist.all_reduce(tl, op=dist.ReduceOp.MAX)
    loop_s = float(tl.item())

    # ------------------------------------------------------------- roofline of the dominant rtti kernel (CUDA events)
    # two eager profiling steps, one per injection regime (every rank executes them: on >1 GPU a step contains the exchange)
    roof = cross = None
    st = states[0]
    prof_idx = sorted({0, n_t - 1}) if cfg["inject_selfattn"] > 0 else [0]
    ops.PROFILE = []
    model.profile_events = {}
    graphs_on, model.use_cuda_graphs = model.use_cuda_graphs, False   # eager so every launch carries its events
    with torch.no_grad():
        for i in prof_idx:
            model.rich_text_step(st, i)
    barrier()
    prof, ops.PROFILE = ops.PROFILE, None
    model.use_cuda_graphs = graphs_on
    breakdown = {}
    with torch.no_grad():
        for i in prof_idx:
            model.profile_events = {}
            model.rich_text_step(st, i)
            barrier()
            tag = "inject_on" if float(timesteps[i]) > (1 - cfg["inject_selfattn"]) * 1000 else "inject_off"
            breakdown[tag] = {k: a.elapsed_time(b) for k, (a, b) in model.profile_events.items()}
    model.profile_events = None
    if rank == 0:
        hbm, tf_burst, tf_sust, src = peaks()
        agg = {}
        for ev0, ev1, kind, flops, nbytes, shape in prof:
            a = agg.setdefault(kind, [0.0, 0.0, 0.0, 0])
            a[0] += ev0.elapsed_time(ev1) * 1e-3; a[1] += flops; a[2] += nbytes; a[3] += 1
        s = agg.get("self")
        c = agg.get("cross")
        n_prof = len(prof_idx)
        if s:
            ach = s[1] / s[0] / 1e12
            traffic, tnote = ncu_traffic("attn_self_kernel")
            roof = {"kernel": "attn_self_kernel<NV> (self-attention, tcgen05/TMEM/TMA, head_dim 64, grouped PV on injection steps)",
                    "bound": "tensor", "achieved": ach, "peak": tf_sust, "unit": "TFLOP/s", "frac": ach / tf_sust,
                    "flops_counted": "algorithmic: QK^T once per score source + PV per entry (what the reference evaluates)",
                    "traffic": traffic, "traffic_note": tnote,
                    "peak_source": f"{src} bf16_tflops_sustained (kernel timed inside a long step)",
                    "launches_timed": s[3], "profiled_steps": n_prof, "ms_per_step_in_kernel": s[0] * 1e3 / n_prof}
        if c:
            gbs = c[2] / c[0] / 1e9
            ctraffic, cnote = ncu_traffic("attn_fwd_kernel_cross")
            cross = {"kernel": "attn_cross_kernel (cross-attention, 77 keys, font-size re-weighting on pass B; persistent, TMA ring + tcgen05/TMEM)", "bound": "hbm", "achieved": gbs,
                     "peak": hbm, "unit": "GB/s", "frac": gbs / hbm, "tensor_tflops": c[1] / c[0] / 1e12,
                     "traffic": ctraffic, "traffic_note": cnote,
                     "launches_timed": c[3], "ms_per_step_in_kernel": c[0] * 1e3 / n_prof}

    if rank != 0:
        return
    steps_per_s = args.steps / (ms * 1e-3)
    e2e_v = args.steps / e2e_s
    line = {
        "metric": "denoising steps/sec", "value": steps_per_s, "unit": "steps/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
        "config": bench_config(args.config),
        "execution": "the passes of a rank run as one batched, CUDA-graph-replayed UNet call",
        "parallelism": (f"UNet passes region-parallel x{world} (fused peer-memory exchange; "
                        + ("pass D on one rank, its Q|K and injected feature pushed to the region-pass ranks over NVLink)"
                           if model.remote_qk and model.fused_exchange else "pass D replicated on the region-pass ranks)")
                        + (f", colour guidance stripe-parallel x{world}" + (" replayed as one CUDA graph" if model.graph_guidance else "")
                           if cfg["color"] else "")
                        + (f"; {cfg['images']} images data-parallel first" if cfg["images"] > 1 else "")
                        if world > 1 else "single GPU"),
        "clocks": clk, "gpu_launches": launches,
        "e2e": {"value": e2e_v, "unit": "steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "last_color_loss": loss,
                "how": "RegionDiffusionXL.rich_text_step per step; all step inputs staged from pinned host memory every step, "
                       "latents + loss copied back every step (async D2H, consumed one step later)"},
        "consistency": {"device_ms_per_step": ms / args.steps, "e2e_ms_per_step": 1000.0 * e2e_s / args.steps,
                        "device_le_e2e": ms / args.steps <= 1.02 * 1000.0 * e2e_s / args.steps},
        "sampling_loop": {"steps": n_t, "wall_s": loop_s, "steps_per_s": n_t * 1.0 / loop_s,
                          "what": f"all {n_t} steps of one rich-text sampling run in schedule order through rich_text_step "
                                  "(inputs from pinned host memory once, latents read back once; CUDA graphs warm)"},
        "roofline": roof, "roofline_cross_attention": cross, "breakdown_ms": breakdown,
        "ranks_bit_identical": ranks_identical, "single_gpu_check": check, "fallback": fallback,
    }
    if world == 1 and not args.no_cpu_baseline:
        pps = passes_per_step(cfg) * cfg["images"]
        times, threads = cpu_oracle_pass_times(cfg["model"], 1, 0)
        v = 1.0 / (pps * times[0])
        line["cpu_baseline"] = {"value": v, "unit": "steps/s", "cores": threads, "kind": "port",
                                "sample": f"ONE WHOLE batch-1 {cfg['model']} UNet pass of the fp32 CPU oracle ({times[0]:.1f} s, cold) x "
                                          f"{pps} passes/step; the VAE colour guidance and the blend are NOT included, so this CPU "
                                          "figure is optimistic (bench.py --impl reference measures the guidance too)"}
        line["gpu_eager_baseline"] = gpu_eager_port(model, cfg, dev)
    print(json.dumps(line), flush=True)


def gpu_eager_port(model, cfg, dev):
    """The reference's algorithm as plain PyTorch-eager on the SAME GPU (SURVEY §8d "honest GPU baseline"): the oracle
    restatement run on the device in fp16 with this model's weights — probabilities materialised, head mean on every
    call, batch-1 passes one after another (models/region_diffusion_sdxl.py:787-821). A baseline leg, never the product."""
    import torch
    from oracle import unet_oracle as uo
    try:
        ocfg = uo.sdxl_config() if cfg["model"] == "sdxl" else uo.sd15_config()
        sd = {k: v for k, v in model.unet.state_dict().items()}
        g = torch.Generator(device=dev).manual_seed(0)
        x = torch.randn(1, 4, 128, 128, generator=g, device=dev).half()
        ctx = torch.randn(1, 77, 2048, generator=g, device=dev).half()
        added = {"text_embeds": torch.randn(1, 1280, generator=g, device=dev).half(),
                 "time_ids": torch.tensor([[1024.0, 1024, 0, 0, 1024, 1024]], device=dev)}
        t = torch.tensor(981.0, device=dev)
        with torch.no_grad():
            uo.unet_forward(sd, ocfg, x, t, ctx, added)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            n = 4
            for _ in range(n):
                uo.unet_forward(sd, ocfg, x, t, ctx, added)
            e1.record()
            torch.cuda.synchronize()
        ms_pass = e0.elapsed_time(e1) / n
        pps = passes_per_step(cfg) * cfg["images"]
        return {"kind": "port (oracle restatement run eagerly on this GPU, fp16, batch-1 passes, probabilities materialised)",
                "ms_per_pass": ms_pass, "passes_per_step": pps, "steps_per_s_unet_only": 1000.0 / (pps * ms_pass)}
    except Exception as e:   # a baseline leg must never take the product line down
        return {"unavailable": repr(e)[:200]}


# ------------------------------------------------------------------------------------------- product arm, SD1.5 configs
def run_product_sd(args, rank, world, local_rank):
    """Configs 1 / 2 (SD1.5 512^2). The PNDM scheduler is stateful across steps, so the timed unit is a whole
    `produce_latents` call of K steps (K + 1 UNet evaluations, as the reference's PLMS does); config 2 additionally
    reports the token-map capture pass (plain CFG, 41 steps) and `get_token_maps`."""
    import torch
    import torch.distributed as dist
    from rtti_b200 import ops
    from rtti_b200.attention_utils import get_token_maps
    from rtti_b200.region_diffusion import RegionDiffusion
    cfg = CONFIGS[args.config]
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    model = RegionDiffusion.from_synthetic(seed=0, device=dev, with_vae=False)
    wl = synth_workload(cfg)
    pinned = {"ctx": wl["ctx"].pin_memory(), "latents": wl["latents"].pin_memory(), "masks": [m.pin_memory() for m in wl["masks"]]}
    tfd = {"word_pos": wl["tfd"]["word_pos"], "font_size": wl["tfd"]["font_size"]} if cfg["regions"] > 1 else {}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def call(steps, src):
        model.masks = [m.to(dev, non_blocking=True) for m in src["masks"]]
        return model.produce_latents(src["ctx"].to(dev, non_blocking=True), num_inference_steps=steps, guidance_scale=GUIDANCE,
                                     latents=src["latents"].to(dev, non_blocking=True), text_format_dict=tfd,
                                     inject_selfattn=cfg["inject_selfattn"], inject_background=cfg["inject_background"])

    dev_src = {"ctx": wl["ctx"].to(dev), "latents": wl["latents"].to(dev), "masks": [m.to(dev) for m in wl["masks"]]}
    extras = {}
    with torch.no_grad():
        call(max(args.warmup, 3), dev_src)
        call(args.steps, dev_src)
        barrier()
        clocks = ClockSampler(local_rank) if rank == 0 else None
        launches0 = ops.LAUNCHES
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = call(args.steps, dev_src)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        launches = ops.LAUNCHES - launches0
        clk = clocks.stop() if clocks else None
        assert bool(torch.isfinite(out.float()).all())
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, {"latents": out})
        host_lat = torch.empty(1, 4, 64, 64, dtype=torch.float16).pin_memory()
        barrier()
        t0 = time.perf_counter()
        out = call(args.steps, pinned)
        host_lat.copy_(out)
        barrier()
        e2e_s = time.perf_counter() - t0
        if args.config == 2 and rank == 0:
            model.register_tokenmap_hooks()
            ctx2 = torch.cat([dev_src["ctx"][:1], dev_src["ctx"][-1:]])
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            model.produce_attn_maps(None, None, num_inference_steps=cfg["schedule"], guidance_scale=GUIDANCE,
                                    latents=dev_src["latents"], text_embeddings=ctx2, decode=False)
            torch.cuda.synchronize()
            extras["capture_pass_s"] = time.perf_counter() - t0
            t0 = time.perf_counter()
            get_token_maps(model.selfattn_maps, model.crossattn_maps, model.n_maps, None, 64, 64,
                           [torch.LongTensor([2]), torch.LongTensor([5, 6])], seed=3, num_segments=9)
            extras["get_token_maps_s"] = time.perf_counter() - t0
            extras["note"] = ("capture pass = plain CFG loop, 41 steps, on-device fp32 token-map accumulation; get_token_maps = device "
                              "averaging/resizes + scikit-learn SpectralClustering(n_init=100) on the host, called once here (sample.py calls it twice)")
            model.remove_tokenmap_hooks()
    t = torch.tensor([ms, e2e_s], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, e2e_s = float(t[0]), float(t[1])
    if rank != 0:
        return
    h2d = sum(x.numel() * x.element_size() for x in [pinned["ctx"], pinned["latents"], *pinned["masks"]])
    line = {"metric": "denoising steps/sec", "value": args.steps / (ms * 1e-3), "unit": "steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f16", "data": "synthetic", "config": bench_config(args.config),
            "execution": "one produce_latents call of K steps (PLMS: K + 1 batched UNet evaluations), eager launches",
            "clocks": clk, "gpu_launches": launches,
            "e2e": {"value": args.steps / e2e_s, "unit": "steps/s", "h2d_bytes_per_step": h2d / args.steps,
                    "d2h_bytes_per_step": host_lat.numel() * 2 / args.steps,
                    "note": "inputs are copied once per sampling call, not per step (the PNDM state couples the steps)"},
            "roofline": None, "token_map_pass": extras or None}
    if world == 1 and not args.no_cpu_baseline:
        pps = passes_per_step(cfg)
        times, threads = cpu_oracle_pass_times("sd15", 2, 1)
        tp = sum(times) / len(times)
        line["cpu_baseline"] = {"value": 1.0 / (pps * tp), "unit": "steps/s", "cores": threads, "kind": "port",
                                "sample": f"2 WHOLE batch-1 SD1.5 UNet passes of the fp32 CPU oracle (mean {tp:.2f} s) x {pps} passes/step"}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", type=int, default=3, choices=sorted(CONFIGS))
    ap.add_argument("--impl", default="rtti", choices=["rtti", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--check", action="store_true", help="N > 1: also compare with a single-GPU run of the same steps")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the product arm (--impl rtti)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if args.warmup < 3:
        args.warmup = 3
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        if CONFIGS[args.config]["model"] == "sdxl":
            run_product_xl(args, rank, world, local_rank)
        else:
            run_product_sd(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
