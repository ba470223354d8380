"""CPU: the oracle and the host-side text preparation against outputs of the UNMODIFIED reference on inputs other
than those of test_oracle_golden.py. The reference outputs were recorded by running the reference on the inputs
defined here (`python -m oracle.gen_golden oracle_vs_reference`) into tests/golden/oracle_vs_reference.npz
(arrays, parameter inventories) and tests/golden/richtext_reference.json (the text-preparation results)."""
import contextlib
import json
import os

import numpy as np
import pytest
import torch

from oracle import unet_oracle as uo

UNET_CASES = [(uo.tiny_sd_config, 3), (uo.tiny_xl_config, 4)]
UNET_TIMESTEPS = (torch.tensor(999), torch.tensor(37.0, dtype=torch.float64))
XL_CASES = [
    (4, 3, 0.4, 0.0, False, True, 71),      # more regions, self-attention / feature injection on the first step only
    (2, 3, 0.0, 0.4, True, False, 72),      # configs[3]-like: background injection only (the joint-stepping quirk), colour guidance
]
XL_SAMPLE = 8192   # latents of an XL case recorded at this many fixed positions (of 65536)


@pytest.fixture(scope="module")
def golden(golden_dir):
    return np.load(os.path.join(golden_dir, "oracle_vs_reference.npz"), allow_pickle=False)


@contextlib.contextmanager
def one_thread():
    """The CPU convolution / GEMM kernels split their reductions by thread count, so a bit-exact comparison with recorded
    outputs holds only at the thread count they were recorded with: one."""
    n = torch.get_num_threads()
    torch.set_num_threads(1)
    try:
        yield
    finally:
        torch.set_num_threads(n)


def inventory(golden, name):
    """{parameter name: shape} of a reference UNet's state_dict, as recorded."""
    return {k: tuple(int(d) for d in s.split(",") if d) for k, s in zip(golden[f"{name}_names"], golden[f"{name}_shapes"])}


def unet_inputs(cfg, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(2, 4, 16, 16, generator=g)
    ctx = torch.randn(2, 77, cfg.cross_attention_dim, generator=g)
    added = None
    if cfg.addition_embed_type:
        pooled = cfg.projection_class_embeddings_input_dim - 6 * cfg.addition_time_embed_dim
        added = {"text_embeds": torch.randn(2, pooled, generator=g), "time_ids": torch.tensor([[128.0, 128, 0, 0, 128, 128]] * 2)}
    return x, ctx, added


def attention_inputs():
    """Seeded weights (nn.Linear's default init range) and inputs of a 2-head cross-attention, query 64, context 48."""
    g = torch.Generator().manual_seed(0)

    def linear(n_out, n_in):
        return (torch.rand(n_out, n_in, generator=g) * 2 - 1) / n_in ** 0.5

    sd = {"a.to_q.weight": linear(64, 64), "a.to_k.weight": linear(64, 48), "a.to_v.weight": linear(64, 48),
          "a.to_out.0.weight": linear(64, 64), "a.to_out.0.bias": linear(1, 64)[0]}
    hs, ctx = torch.randn(1, 32, 64, generator=g), torch.randn(1, 77, 48, generator=g)
    aw = {"word_pos": torch.LongTensor([1, 4, 4]), "font_size": torch.FloatTensor([3.0, -2.0, 0.25])}
    return sd, hs, ctx, aw


def xl_sample_index():
    return np.random.RandomState(0).permutation(4 * 128 * 128)[:XL_SAMPLE]


@pytest.mark.parametrize("cfg_fn,seed", UNET_CASES)
def test_unet_forward_bit_exact(golden, cfg_fn, seed):
    cfg = cfg_fn()
    sd = uo.make_state_dict(cfg, seed)
    name = cfg_fn.__name__
    assert inventory(golden, name) == {k: tuple(v.shape) for k, v in sd.items()}
    assert inventory(golden, name) == {k: tuple(v) for k, v in uo.param_shapes(cfg).items()}
    x, ctx, added = unet_inputs(cfg, seed)
    with torch.no_grad(), one_thread():
        for i, t in enumerate(UNET_TIMESTEPS):
            yr = torch.from_numpy(golden[f"{name}_out{i}"])
            yo = uo.unet_forward(sd, cfg, x, t, ctx, added)
            assert torch.equal(yr, yo)


def test_full_size_parameter_inventories(golden):
    for cfg_fn, nparams in ((uo.sd15_config, 859.5e6), (uo.sdxl_config, 2567.5e6)):
        shapes = inventory(golden, cfg_fn.__name__)
        mine = {k: tuple(v) for k, v in uo.param_shapes(cfg_fn()).items()}
        assert shapes == mine
        assert abs(sum(torch.Size(s).numel() for s in mine.values()) - nparams) < 0.1e6


def test_attention_fontsize_and_injection(golden):
    sd, hs, ctx, aw = attention_inputs()

    class C(uo.AttnControl):
        def pre_attn(self, name):
            return None, aw

        def post_attn(self, name, pavg, p):
            self.out = (pavg, p)

    c = C()
    o_ref, pavg_ref, p_ref = (torch.from_numpy(golden[k]) for k in ("attn_out", "attn_pavg", "attn_probs"))
    with torch.no_grad():
        o = uo.attention(sd, "a", 2, hs, ctx, c)
    assert torch.allclose(o, o_ref, atol=1e-6) and torch.allclose(c.out[0], pavg_ref, atol=1e-7)
    assert torch.allclose(c.out[1], p_ref, atol=1e-7)


# --------------------------------------------------------------------------- host-side text preparation (SURVEY 8f.4)
class _Tok:
    def _tokenize(self, text):
        return text.lower().replace(",", " ,").split()


class _Model:
    tokenizer = _Tok()


_DELTAS = [
    {"ops": [{"insert": "a church "}, {"attributes": {"color": "#fd6c9e"}, "insert": "garden"},
             {"insert": " with "}, {"attributes": {"font": "slabo"}, "insert": "mountains"},
             {"attributes": {"size": "60px"}, "insert": " snowy"}, {"attributes": {"link": "a red sun"}, "insert": " sky"},
             {"insert": "\n"}]},
    {"ops": [{"attributes": {"font": "mirza"}, "insert": "a lake"}, {"attributes": {"font": "mirza"}, "insert": " at dawn"},
             {"insert": ", "}, {"attributes": {"color": "#00ff00", "size": "18px", "strike": True}, "insert": "reeds"},
             {"insert": " and a "}, {"attributes": {"color": "#a52a2a"}, "insert": "boat"}, {"insert": "\n"}]},
    {"ops": [{"insert": "a plain prompt without attributes\n"}]},
]


def to_json(x):
    """Nested lists / tuples / dicts of tensors and scalars -> JSON-able (tensors tagged with dtype and shape)."""
    if torch.is_tensor(x):
        return {"tensor": x.tolist(), "dtype": str(x.dtype).replace("torch.", ""), "shape": list(x.shape)}
    if isinstance(x, (list, tuple)):
        return [to_json(y) for y in x]
    if isinstance(x, dict):
        return {k: to_json(v) for k, v in x.items()}
    return x


def from_json(x):
    if isinstance(x, dict) and set(x) == {"tensor", "dtype", "shape"}:
        return torch.tensor(x["tensor"], dtype=getattr(torch, x["dtype"])).reshape(x["shape"])
    if isinstance(x, list):
        return [from_json(y) for y in x]
    if isinstance(x, dict):
        return {k: from_json(v) for k, v in x.items()}
    return x


@pytest.mark.parametrize("delta", _DELTAS)
def test_richtext_utils_match_the_reference_functions(golden_dir, delta):
    """rtti_b200.richtext_utils against utils/richtext_utils.py of the unmodified reference on the same Quill deltas:
    parse_json :74-136, get_region_diffusion_input :139-185, get_attention_control_input :188-209,
    get_gradient_guidance_input :212-234 — identical prompts, token ids, font sizes and target colours."""
    from rtti_b200 import richtext_utils as ru
    with open(os.path.join(golden_dir, "richtext_reference.json")) as f:
        rec = next(r for r in json.load(f) if r["delta"] == delta)

    def same(a, b):
        if torch.is_tensor(a) or torch.is_tensor(b):
            return torch.is_tensor(a) and torch.is_tensor(b) and a.shape == b.shape and torch.allclose(a.float().cpu(), b.float().cpu())
        if isinstance(a, (list, tuple)):
            return isinstance(b, (list, tuple)) and len(a) == len(b) and all(same(x, y) for x, y in zip(a, b))
        return a == b

    out_r = from_json(rec["parse_json"])
    out_p = ru.parse_json(delta, device="cpu")
    assert len(out_r) == len(out_p) == 9
    for i, (a, b) in enumerate(zip(out_r, out_p)):
        assert same(a, b), f"parse_json output {i}: {a!r} vs {b!r}"
    base, styles, notes, note_t, cspans, cnames, crgbs, sizes, use_grad = out_r
    pr, idr, btr = from_json(rec["region_diffusion_input"])
    pp, idp, btp = ru.get_region_diffusion_input(_Model(), base, styles, notes, note_t, cspans, cnames)
    assert pr == pp and btr == btp and same(idr, idp)
    tr = from_json(rec["attention_control_input"])
    tp = ru.get_attention_control_input(_Model(), btp, sizes, device="cpu")
    assert set(tr) == set(tp) and all(same(tr[k], tp[k]) for k in tr)
    tr2, cr = from_json(rec["gradient_guidance_input"])
    tp2, cp = ru.get_gradient_guidance_input(_Model(), btp, cspans, out_p[6], dict(tp), color_guidance_weight=0.5)
    assert same(cr, cp) and set(tr2) == set(tp2)
    for k in tr2:
        assert same(tr2[k], tp2[k]), k


@pytest.mark.parametrize("n_prompts,steps,inject_selfattn,inject_background,use_guidance,with_fs,seed", XL_CASES)
def test_xl_rich_loop_live_reference_other_settings(golden, n_prompts, steps, inject_selfattn, inject_background, use_guidance,
                                                    with_fs, seed):
    """RegionDiffusionXL.sample(run_rich_text=True) of the UNMODIFIED reference (models/region_diffusion_sdxl.py:772-878)
    against the oracle's rich_text_loop at settings the committed fixtures do not cover: other region counts, step
    counts, injection windows, with / without font sizes and colour guidance. The reference's latents are recorded at
    XL_SAMPLE fixed random positions."""
    from oracle import gen_golden as gg, sampler_oracle as sam, schedulers_oracle as so
    from tests import synth
    case = XL_CASES.index((n_prompts, steps, inject_selfattn, inject_background, use_guidance, with_fs, seed))
    cfg = uo.tiny_xl_config()
    S = 128   # the reference asserts a 64-wide injected feature map (sdxl.py:1090): 1024^2 images only
    inp = gg.synth_inputs(cfg, n_prompts, S, seed)
    ctx, te = inp["ctx"], inp["text_embeds"]
    tfd = gg.text_format(1, S, seed, with_fs=with_fs)
    if use_guidance:
        tfd.update(gg.color_dict(inp["masks"], S, weight=0.7))
    out = torch.from_numpy(golden[f"xl{case}_latents_sample"])
    sd = uo.make_state_dict(cfg, 5)
    sch = so.EulerDiscreteSchedulerOracle()
    sch.set_timesteps(steps)
    added = {"text_embeds": te, "time_ids": inp["time_ids"]}
    lat = sam.rich_text_loop(sam.make_unet_fn(sd, cfg), sch, ctx, inp["masks"], inp["latents"].clone() * sch.init_noise_sigma,
                             steps, 6.0, xl=True, added_cond=added, use_guidance=use_guidance, text_format_dict=dict(tfd),
                             inject_selfattn=inject_selfattn, inject_background=inject_background,
                             vae_decode=synth.TinyVAE() if use_guidance else None, scaling_factor=0.13025)
    assert lat.shape == (1, 4, S, S)
    assert torch.isfinite(out).all() and torch.isfinite(lat).all()
    torch.testing.assert_close(lat.flatten()[torch.from_numpy(xl_sample_index())], out, atol=5e-4, rtol=1e-4)
