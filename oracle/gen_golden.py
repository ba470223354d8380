"""TEST INFRASTRUCTURE — generates tests/golden/*.npz by running the UNMODIFIED reference
(/root/reference, imported through oracle/ref_shim.py) on seeded synthetic inputs.

Run in the build container (the reference tree does not exist on the GPU box):
    python -m oracle.gen_golden            # all fixtures
The fixtures pin (a) the oracle restatement (tests/test_oracle_golden.py, CPU) and (b) the CUDA product
path (tests/test_parity_gpu.py, GPU). Weights are never stored: both sides rebuild them with
oracle.unet_oracle.make_state_dict(cfg, seed). The two schedulers are the restated third-party ones
(oracle/schedulers_oracle.py) on both arms — diffusers is not installed.
"""
import json
import os
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, ROOT)

import torchvision  # noqa: F401,E402  (must be imported before the stubs are installed)

from oracle import ref_shim, schedulers_oracle as so, unet_oracle as uo  # noqa: E402


def synth_inputs(cfg, n_prompts, latent, seed):
    """Seeded inputs shared by fixtures and tests: latents, per-prompt contexts (+ SDXL added conds), masks."""
    g = torch.Generator().manual_seed(seed)
    lat = torch.randn(1, 4, latent, latent, generator=g)
    ctx = torch.randn(n_prompts + 1, 77, cfg.cross_attention_dim, generator=g)
    out = {"latents": lat, "ctx": ctx}
    if cfg.addition_embed_type:
        pooled = cfg.projection_class_embeddings_input_dim - 6 * cfg.addition_time_embed_dim
        out["text_embeds"] = torch.randn(n_prompts + 1, pooled, generator=g)
        s = float(latent * 8)
        out["time_ids"] = torch.tensor([[s, s, 0.0, 0.0, s, s]])
    # smooth random partition of the latent grid into n_prompts soft masks that sum to 1
    logits = torch.randn(n_prompts, 1, 8, 8, generator=g)
    up = torch.nn.functional.interpolate(logits, (latent, latent), mode="bicubic", align_corners=False)
    m = torch.softmax(up * 3.0, dim=0)
    out["masks"] = [m[i:i + 1].repeat(1, 4, 1, 1) for i in range(n_prompts)]
    return out


def text_format(n_colors, latent, seed, with_fs=True):
    g = torch.Generator().manual_seed(seed + 1000)
    tfd = {"word_pos": None, "font_size": None}
    if with_fs:
        tfd["word_pos"] = torch.LongTensor([2, 5, 9])
        tfd["font_size"] = torch.FloatTensor([2.0, 0.5, -1.5])
    return tfd


def ref_unet(ns, cfg, seed):
    unet = ns.unet_2d_condition.UNet2DConditionModel(**cfg.ref_kwargs())
    unet.load_state_dict(uo.make_state_dict(cfg, seed))
    return unet.eval()


def gen_unet(ns):
    for name, cfg, S in (("tiny_sd", uo.tiny_sd_config(), 16), ("tiny_xl", uo.tiny_xl_config(), 16)):
        unet = ref_unet(ns, cfg, 0)
        inp = synth_inputs(cfg, 1, S, 11)
        x = torch.cat([inp["latents"], inp["latents"].flip(-1)])
        added = None
        if cfg.addition_embed_type:
            added = {"text_embeds": inp["text_embeds"], "time_ids": inp["time_ids"].repeat(2, 1)}
        with torch.no_grad():
            y = unet(x, torch.tensor(481), encoder_hidden_states=inp["ctx"], added_cond_kwargs=added)["sample"]
        np.savez_compressed(os.path.join(GOLD, f"unet_{name}.npz"), out=y.numpy(), weight_seed=0, input_seed=11,
                            latent=S, timestep=481)
        print("unet", name, float(y.abs().mean()))


def gen_attention(ns):
    """Reference Attention module: plain, font-size, injected probabilities, head average."""
    torch.manual_seed(3)
    A = ns.attention_processor.Attention
    res = {}
    for tag, C, heads, ctxd, T in (("cross", 128, 4, 96, 64), ("self", 128, 4, None, 64)):
        attn = A(query_dim=C, cross_attention_dim=ctxd, heads=heads, dim_head=C // heads, bias=False)
        sd = {k: v.clone() for k, v in attn.state_dict().items()}
        hs = torch.randn(2, T, C)
        ctx = torch.randn(2, 77, ctxd) if ctxd else None
        with torch.no_grad():
            o, (pavg, p) = attn(hs, encoder_hidden_states=ctx)
            res[f"{tag}_hs"] = hs.numpy(); res[f"{tag}_out"] = o.numpy(); res[f"{tag}_pavg"] = pavg.numpy()
            if ctx is not None:
                res[f"{tag}_ctx"] = ctx.numpy()
                aw = {"word_pos": torch.LongTensor([2, 5, 5, 9]), "font_size": torch.FloatTensor([2.0, 0.5, 3.0, -1.5])}
                o2, (pavg2, p2) = attn(hs, None, aw, encoder_hidden_states=ctx)
                res[f"{tag}_fs_out"] = o2.numpy(); res[f"{tag}_fs_pavg"] = pavg2.numpy()
            else:
                hs2 = torch.randn(2, T, C)
                o3, _ = attn(hs2, p)  # real_attn_probs injection
                res[f"{tag}_inj_hs"] = hs2.numpy(); res[f"{tag}_inj_out"] = o3.numpy()
        for k, v in sd.items():
            res[f"{tag}_w_{k}"] = v.numpy()
    np.savez_compressed(os.path.join(GOLD, "attention.npz"), **res)
    print("attention ok")


def make_sd_sampler(ns, cfg, seed):
    RD = ns.region_diffusion.RegionDiffusion
    m = RD.__new__(RD)
    torch.nn.Module.__init__(m)
    m.device = "cpu"
    m.unet = ref_unet(ns, cfg, seed)
    m.scheduler = so.PNDMSchedulerOracle()
    m.alphas_cumprod = m.scheduler.alphas_cumprod
    m.masks = []
    m.color_loss = torch.nn.functional.mse_loss
    m.forward_hooks, m.forward_replacement_hooks = [], []
    return m


class _TinyVAE:
    """Differentiable stand-in for AutoencoderKL.decode used ONLY to exercise the colour-guidance arithmetic
    (the real VAE is third-party and needs weights): nearest x8 upsample of a fixed 1x1 conv 4->3."""

    def __init__(self):
        g = torch.Generator().manual_seed(77)
        self.w = torch.randn(3, 4, 1, 1, generator=g) * 0.5
        self.config = types.SimpleNamespace(scaling_factor=0.13025, block_out_channels=(1, 1, 1, 1))
        self.decoder = types.SimpleNamespace(mid_block=types.SimpleNamespace(attentions=[types.SimpleNamespace(processor=None)]))
        self.post_quant_conv = types.SimpleNamespace(to=lambda *a, **k: None)

    def to(self, *a, **k):
        return self

    def decode(self, z, return_dict=True):
        img = torch.nn.functional.interpolate(torch.nn.functional.conv2d(z, self.w.to(z.dtype)), scale_factor=8.0, mode="nearest")
        return types.SimpleNamespace(sample=img)


def color_dict(masks, latent, weight=1.0):
    """text_format_dict entries of utils/richtext_utils.py:212-234 for one coloured region (region 0)."""
    up = torch.nn.functional.interpolate(masks[0], (latent * 8, latent * 8), mode="bicubic", antialias=True).clamp(0, 1)
    return {"target_RGB": [torch.tensor([0.99, 0.42, 0.62]).reshape(1, 3, 1, 1)], "guidance_start_step": 999,
            "color_guidance_weight": weight, "color_obj_atten": [up], "color_obj_atten_all": masks[0].clone()}


def gen_sd_loops(ns):
    cfg = uo.tiny_sd_config()
    S = 64
    m = make_sd_sampler(ns, cfg, 1)
    inp = synth_inputs(cfg, 3, S, 21)
    # --- plain CFG pass with token-map capture (12 steps -> 13 evaluations, capture from the 11th call)
    m.register_tokenmap_hooks()
    m.get_text_embeds = lambda p, n: torch.cat([inp["ctx"][:1], inp["ctx"][-1:]])
    m.decode_latents = lambda lat: torch.zeros(1, 3, 8, 8)
    m._plain_latents = None
    orig_step = m.scheduler.step
    m.produce_attn_maps(["x"], [""], height=S * 8, width=S * 8, num_inference_steps=12, guidance_scale=8.5,
                        latents=inp["latents"].clone())
    selfm = {k: v.clone() for k, v in m.selfattn_maps.items()}
    crossm = {k: v.clone() for k, v in m.crossattn_maps.items()}
    nmaps = dict(m.n_maps)
    m.remove_tokenmap_hooks()
    from oracle import token_maps_oracle as tmo
    aff = tmo.self_affinity(selfm)
    cross = tmo.cross_maps_mean(crossm)
    res = {"plain_aff_rows": aff[::64], "plain_cross_mean": cross,
           "plain_self_names": np.array(sorted(selfm.keys())), "plain_cross_names": np.array(sorted(crossm.keys())),
           "plain_ncalls": nmaps[sorted(nmaps.keys())[0]],
           "plain_self_rowsum": np.array([float(selfm[k][0, 0].sum()) for k in sorted(selfm.keys())]),
           "plain_cross_rowsum": np.array([float(crossm[k][0, 0].sum()) for k in sorted(crossm.keys())])}
    # --- rich-text loop: 3 regions, font sizes, self-attn + background injection, colour guidance
    m.masks = inp["masks"]
    m.vae = _TinyVAE()
    tfd = text_format(1, S, 21)
    tfd.update(color_dict(inp["masks"], S, weight=0.5))
    lat = m.produce_latents(inp["ctx"], height=S * 8, width=S * 8, num_inference_steps=4, guidance_scale=8.5,
                            latents=inp["latents"].clone(), use_guidance=True, text_format_dict=tfd,
                            inject_selfattn=0.3, inject_background=0.5)
    res["rich_latents"] = lat.detach().numpy()
    m.scheduler = so.PNDMSchedulerOracle()
    lat2 = m.produce_latents(inp["ctx"], height=S * 8, width=S * 8, num_inference_steps=3, guidance_scale=8.5,
                             latents=inp["latents"].clone(), use_guidance=False, text_format_dict={"word_pos": None, "font_size": None},
                             inject_selfattn=0, inject_background=0)
    res["rich_noinject_latents"] = lat2.detach().numpy()
    np.savez_compressed(os.path.join(GOLD, "sd_loops.npz"), **res)
    print("sd loops ok", float(lat.abs().mean()), float(lat2.abs().mean()))


def make_xl_sampler(ns, cfg, seed, embeds):
    X = ns.region_diffusion_sdxl.RegionDiffusionXL
    m = X.__new__(X)
    m.unet = ref_unet(ns, cfg, seed)
    m.scheduler = so.EulerDiscreteSchedulerOracle()
    m.vae = _TinyVAE()
    m.vae_scale_factor = 8
    m.default_sample_size = 128
    pooled = cfg.projection_class_embeddings_input_dim - 6 * cfg.addition_time_embed_dim
    m.text_encoder_2 = types.SimpleNamespace(config=types.SimpleNamespace(projection_dim=pooled), dtype=torch.float32)
    m.masks = []
    m.color_loss = torch.nn.functional.mse_loss
    m.forward_hooks, m.forward_replacement_hooks = [], []
    m.encode_prompt = lambda *a, **k: embeds
    m.check_inputs = lambda *a, **k: None
    X._execution_device = property(lambda self: torch.device("cpu"))

    class _PB:
        def __enter__(self): return self
        def __exit__(self, *a): return False
        def update(self): pass

    m.progress_bar = lambda total=None: _PB()
    return m


def gen_xl_loops(ns):
    if ns.region_diffusion_sdxl is None:
        raise RuntimeError(ns.region_diffusion_sdxl_error)
    cfg = uo.tiny_xl_config()
    S = 128
    inp = synth_inputs(cfg, 3, S, 31)
    ctx, te = inp["ctx"], inp["text_embeds"]
    res = {}
    # plain pass (batch 2, capture): embeds = (prompt, negative, pooled, negative pooled)
    m = make_xl_sampler(ns, cfg, 2, (ctx[-1:], ctx[:1], te[-1:], te[:1]))
    m.register_tokenmap_hooks()
    lat0 = inp["latents"].clone()
    out = m.sample(["x"], height=S * 8, width=S * 8, num_inference_steps=12, guidance_scale=8.5, negative_prompt=[""],
                   latents=lat0, output_type="latent", run_rich_text=False)
    res["plain_latents"] = out.images.numpy()
    selfm = {k: v.clone() for k, v in m.selfattn_maps.items()}
    crossm = {k: v.clone() for k, v in m.crossattn_maps.items()}
    from oracle import token_maps_oracle as tmo
    res["plain_aff_rows"] = tmo.self_affinity(selfm)[::64]
    res["plain_cross_names"] = np.array(sorted(crossm.keys()))
    if crossm:
        res["plain_cross_mean"] = tmo.cross_maps_mean(crossm)
    res["plain_self_rowsum"] = np.array([float(selfm[k][0, 0].sum()) for k in sorted(selfm.keys())])
    m.remove_tokenmap_hooks()
    # rich loop
    m = make_xl_sampler(ns, cfg, 2, (ctx[1:], ctx[:1], te[1:], te[:1]))
    m.masks = inp["masks"]
    tfd = text_format(1, S, 31)
    tfd.update(color_dict(inp["masks"], S, weight=1.0))
    out = m.sample(["a", "b", "c"], height=S * 8, width=S * 8, num_inference_steps=4, guidance_scale=8.5,
                   negative_prompt=[""], latents=inp["latents"].clone(), output_type="latent", use_guidance=True,
                   inject_selfattn=0.5, inject_background=0.5, text_format_dict=tfd, run_rich_text=True)
    res["rich_latents"] = out.images.detach().numpy()
    m = make_xl_sampler(ns, cfg, 2, (ctx[1:], ctx[:1], te[1:], te[:1]))
    m.masks = inp["masks"]
    out = m.sample(["a", "b", "c"], height=S * 8, width=S * 8, num_inference_steps=4, guidance_scale=8.5,
                   negative_prompt=[""], latents=inp["latents"].clone(), output_type="latent", use_guidance=False,
                   inject_selfattn=0.0, inject_background=0.5, text_format_dict={"word_pos": None, "font_size": None},
                   run_rich_text=True)
    res["rich_bgonly_latents"] = out.images.detach().numpy()
    np.savez_compressed(os.path.join(GOLD, "xl_loops.npz"), **res)
    print("xl loops ok", {k: float(np.abs(v).mean()) for k, v in res.items() if v.dtype.kind == "f"})


def gen_xl_labels(ns):
    """Segment labels and region masks the reference's get_token_maps (utils/attention_utils.py:233-341) produces from
    the maps its OWN plain pass captures (tiny XL config, same inputs as gen_xl_loops): pins the whole token-map path of
    the product — on-device fp32 capture, averaging, resizes, the host clustering call — down to the label image."""
    cfg = uo.tiny_xl_config()
    S = 128
    inp = synth_inputs(cfg, 3, S, 31)
    ctx, te = inp["ctx"], inp["text_embeds"]
    m = make_xl_sampler(ns, cfg, 2, (ctx[-1:], ctx[:1], te[-1:], te[:1]))
    m.register_tokenmap_hooks()
    m.sample(["x"], height=S * 8, width=S * 8, num_inference_steps=12, guidance_scale=8.5, negative_prompt=[""],
             latents=inp["latents"].clone(), output_type="latent", run_rich_text=False)
    au = ns.attention_utils
    rec = {}
    orig = au.SpectralClustering

    class Recording(orig):
        def fit_predict(self, X, y=None):
            rec["affinity"] = np.array(X)
            rec["labels"] = super().fit_predict(X, y)
            return rec["labels"]

    au.SpectralClustering = Recording
    os.makedirs("/tmp/rtti_golden_tm", exist_ok=True)
    obj = [torch.LongTensor([3]), torch.LongTensor([7, 8])]
    try:
        masks = au.get_token_maps(m.selfattn_maps, m.crossattn_maps, m.n_maps, "/tmp/rtti_golden_tm", S, S, obj, seed=6,
                                  segment_threshold=0.3, num_segments=4)
    finally:
        au.SpectralClustering = orig
    m.remove_tokenmap_hooks()
    np.savez_compressed(os.path.join(GOLD, "xl_token_labels.npz"), labels=rec["labels"].reshape(32, 32).astype(np.int32),
                        masks=torch.cat(masks)[:, 0].numpy(), affinity_rows=rec["affinity"][::64])
    print("xl labels ok", np.bincount(rec["labels"]), [float(x.mean()) for x in masks])


def synth_maps(seed):
    """Synthetic capture dicts with a clear 4-blob structure at 32x32 (+ a 16x16 layer that must be ignored)."""
    g = torch.Generator().manual_seed(seed)
    yy, xx = torch.meshgrid(torch.arange(32.0), torch.arange(32.0), indexing="ij")
    blob = ((yy >= 16).long() * 2 + (xx >= 16).long()).reshape(-1)  # 4 quadrants
    selfm, crossm = {}, {}
    for li in range(3):
        same = (blob[:, None] == blob[None, :]).float()
        a = same * 1.0 + 0.05 * torch.rand(1024, 1024, generator=g)
        a = a / a.sum(-1, keepdim=True)
        selfm[f"l{li}.attn1"] = a[None]
    selfm["small.attn1"] = torch.rand(1, 256, 256, generator=g)
    for li, r in enumerate((32, 16)):
        yy2, xx2 = torch.meshgrid(torch.arange(float(r)), torch.arange(float(r)), indexing="ij")
        q = ((yy2 >= r // 2).long() * 2 + (xx2 >= r // 2).long()).reshape(-1)
        c = 0.01 * torch.rand(1, r * r, 77, generator=g)
        c[0, q == 0, 3] += 0.6
        c[0, q == 3, 7] += 0.5
        c[0, q == 3, 8] += 0.4
        crossm[f"c{li}.attn2"] = c
    return selfm, crossm


def gen_token_maps(ns):
    selfm, crossm = synth_maps(5)
    obj = [torch.LongTensor([3]), torch.LongTensor([7, 8])]
    os.makedirs("/tmp/rtti_golden_tm", exist_ok=True)
    masks = ns.attention_utils.get_token_maps(selfm, crossm, None, "/tmp/rtti_golden_tm", 64, 64, obj, seed=6,
                                              segment_threshold=0.3, num_segments=4)
    np.savez_compressed(os.path.join(GOLD, "token_maps.npz"), masks=torch.cat(masks).numpy(), map_seed=5)
    print("token maps ok", [float(x.mean()) for x in masks])


def gen_oracle_vs_reference(ns):
    """Reference outputs on the inputs tests/test_oracle_vs_reference.py defines: UNet outputs and parameter
    inventories, one font-size attention call, the text preparation of the Quill deltas, XL rich-text loops."""
    from tests import test_oracle_vs_reference as t
    res = {}

    def inventory(name, model):
        sd = model.state_dict()
        res[f"{name}_names"] = np.array(list(sd))
        res[f"{name}_shapes"] = np.array([",".join(str(d) for d in v.shape) for v in sd.values()])

    for cfg_fn, seed in t.UNET_CASES:
        cfg = cfg_fn()
        model = ns.unet_2d_condition.UNet2DConditionModel(**cfg.ref_kwargs())
        model.load_state_dict(uo.make_state_dict(cfg, seed))
        inventory(cfg_fn.__name__, model)
        x, ctx, added = t.unet_inputs(cfg, seed)
        with torch.no_grad(), t.one_thread():
            for i, ts in enumerate(t.UNET_TIMESTEPS):
                res[f"{cfg_fn.__name__}_out{i}"] = model(x, ts, encoder_hidden_states=ctx, added_cond_kwargs=added)["sample"].numpy()
    for cfg_fn in (uo.sd15_config, uo.sdxl_config):
        with torch.device("meta"):
            inventory(cfg_fn.__name__, ns.unet_2d_condition.UNet2DConditionModel(**cfg_fn().ref_kwargs()))

    attn = ns.attention_processor.Attention(query_dim=64, cross_attention_dim=48, heads=2, dim_head=32)
    sd, hs, ctx, aw = t.attention_inputs()
    attn.load_state_dict({k[len("a."):]: v for k, v in sd.items()})
    with torch.no_grad():
        o, (pavg, p) = attn(hs, None, aw, encoder_hidden_states=ctx)
    res.update(attn_out=o.numpy(), attn_pavg=pavg.numpy(), attn_probs=p.numpy())

    rr = ns.richtext_utils
    records = []
    for delta in t._DELTAS:
        out = rr.parse_json(delta)
        base, styles, notes, note_t, cspans, cnames, crgbs, sizes, use_grad = out
        rdi = rr.get_region_diffusion_input(t._Model(), base, styles, notes, note_t, cspans, cnames)
        aci = rr.get_attention_control_input(t._Model(), rdi[2], sizes)
        ggi = rr.get_gradient_guidance_input(t._Model(), rdi[2], cspans, crgbs, dict(aci), color_guidance_weight=0.5)
        records.append({"delta": delta, "parse_json": t.to_json(out), "region_diffusion_input": t.to_json(rdi),
                        "attention_control_input": t.to_json(aci), "gradient_guidance_input": t.to_json(ggi)})
    with open(os.path.join(GOLD, "richtext_reference.json"), "w") as f:
        json.dump(records, f, indent=1)
        f.write("\n")

    if ns.region_diffusion_sdxl is None:
        raise RuntimeError(ns.region_diffusion_sdxl_error)
    cfg = uo.tiny_xl_config()
    S = 128
    for case, (n_prompts, steps, inject_selfattn, inject_background, use_guidance, with_fs, seed) in enumerate(t.XL_CASES):
        inp = synth_inputs(cfg, n_prompts, S, seed)
        ctx, te = inp["ctx"], inp["text_embeds"]
        m = make_xl_sampler(ns, cfg, 5, (ctx[1:], ctx[:1], te[1:], te[:1]))
        m.masks = inp["masks"]
        tfd = text_format(1, S, seed, with_fs=with_fs)
        if use_guidance:
            tfd.update(color_dict(inp["masks"], S, weight=0.7))
        out = m.sample(["p"] * n_prompts, height=S * 8, width=S * 8, num_inference_steps=steps, guidance_scale=6.0,
                       negative_prompt=[""], latents=inp["latents"].clone(), output_type="latent", use_guidance=use_guidance,
                       inject_selfattn=inject_selfattn, inject_background=inject_background, text_format_dict=dict(tfd),
                       run_rich_text=True).images.detach()
        assert out.shape == (1, 4, S, S) and torch.isfinite(out).all()
        res[f"xl{case}_latents_sample"] = out.flatten().numpy()[t.xl_sample_index()]
    np.savez_compressed(os.path.join(GOLD, "oracle_vs_reference.npz"), **res)
    print("oracle vs reference ok", {k: float(np.abs(v).mean()) for k, v in res.items() if v.dtype.kind == "f"})


def main():
    os.makedirs(GOLD, exist_ok=True)
    ns = ref_shim.import_reference()
    which = sys.argv[1:] or ["unet", "attention", "token_maps", "sd", "xl", "xl_labels", "oracle_vs_reference"]
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    if "unet" in which: gen_unet(ns)
    if "attention" in which: gen_attention(ns)
    if "token_maps" in which: gen_token_maps(ns)
    if "sd" in which: gen_sd_loops(ns)
    if "xl" in which: gen_xl_loops(ns)
    if "xl_labels" in which: gen_xl_labels(ns)
    if "oracle_vs_reference" in which: gen_oracle_vs_reference(ns)


if __name__ == "__main__":
    main()
