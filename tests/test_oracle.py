"""CPU tests that pin the oracle (oracle/unet.py, oracle/ddim.py) — the reference has no tests of its own
(SURVEY.md §4), so the restatement is pinned by known answers of the published architecture and by the golden
vectors produced with the reference's own unmodified lora.py / train_util.py (tests/golden/make_golden*.py)."""
import gzip
import json
import os

import pytest
import torch

from conftest import c3lier
from oracle import ddim as oddim
from oracle import port
from oracle import unet as ounet
from sliders_b200 import synthetic

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def _reference_lora_keys():
    """What the reference's LoRANetwork (lora.py) builds on the oracle UNet (tests/golden/make_golden_reference.py)."""
    with gzip.open(os.path.join(GOLDEN, "reference_lora_keys.json.gz"), "rt") as f:
        return json.load(f)


# ---------------------------------------------------------------------------------------- structure KATs
@pytest.mark.parametrize("name,count", [("sdxl", 2_567_463_684), ("sd15", 859_520_964)])
def test_param_count_known_answer(name, count):
    with torch.device("meta"):
        m = ounet.UNet2DConditionModel(getattr(ounet.UNetConfig, name)())
    assert ounet.count_params(m) == count


def test_hf_key_names():
    with torch.device("meta"):
        m = ounet.UNet2DConditionModel(ounet.UNetConfig.sdxl())
    keys = set(m.state_dict().keys())
    for k in ("conv_in.weight", "time_embedding.linear_1.weight", "add_embedding.linear_2.bias",
              "down_blocks.0.resnets.0.time_emb_proj.weight", "down_blocks.0.downsamplers.0.conv.weight",
              "down_blocks.1.attentions.0.transformer_blocks.1.attn1.to_q.weight",
              "down_blocks.2.attentions.1.transformer_blocks.9.ff.net.0.proj.weight",
              "down_blocks.1.attentions.0.proj_in.weight", "mid_block.attentions.0.transformer_blocks.9.attn2.to_out.0.bias",
              "mid_block.resnets.1.conv2.weight", "up_blocks.0.upsamplers.0.conv.weight",
              "up_blocks.2.resnets.2.conv_shortcut.weight", "up_blocks.0.attentions.2.transformer_blocks.0.norm3.weight",
              "conv_norm_out.weight", "conv_out.bias"):
        assert k in keys, k
    assert m.state_dict()["up_blocks.0.resnets.2.conv1.weight"].shape == (1280, 1920, 3, 3)
    assert m.state_dict()["up_blocks.1.resnets.0.conv1.weight"].shape == (640, 1920, 3, 3)
    assert m.state_dict()["down_blocks.1.attentions.0.proj_in.weight"].shape == (640, 640)  # linear projection
    with torch.device("meta"):
        sd1 = ounet.UNet2DConditionModel(ounet.UNetConfig.sd15())
    assert sd1.state_dict()["down_blocks.0.attentions.0.proj_in.weight"].shape == (320, 320, 1, 1)  # conv projection


@pytest.mark.parametrize("name,n_leaves,n_params,rank", [("sdxl", 346, 4_320_000, 4), ("sdxl", 346, 8_640_000, 8),
                                                         ("sd15", 150, 2_906_880, 4)])
def test_reference_lora_injection_counts(name, n_leaves, n_params, rank):
    """The reference's LoRANetwork finds the published adaptor set on the oracle UNet, and the CPU port of its hook
    (oracle/port.py) finds the same leaves in the same order."""
    ref = _reference_lora_keys()["counts"][f"{name}/{rank}"]
    assert ref["n_leaves"] == n_leaves and len(ref["lora_names"]) == n_leaves
    assert ref["n_params"] == n_params
    names = set(ref["lora_names"])
    for k in ("lora_unet_down_blocks_0_resnets_0_conv1", "lora_unet_down_blocks_0_resnets_0_time_emb_proj",
              "lora_unet_down_blocks_0_downsamplers_0_conv", "lora_unet_up_blocks_2_resnets_2_conv_shortcut",
              "lora_unet_mid_block_attentions_0_transformer_blocks_0_attn1_to_out_0"):
        if name == "sdxl":
            assert k in names, k
    assert not any("attn2" in n for n in names)
    with torch.device("meta"):
        m = ounet.UNet2DConditionModel(getattr(ounet.UNetConfig, name)())
        net = port.LoRAHooks(m, rank=rank, alpha=1.0, c3lier=True)
    assert [l.lora_name for l in net.unet_loras] == ref["lora_names"]
    assert sum(p.numel() for p in net.parameters()) == n_params


# ---------------------------------------------------------------------------------------- scheduler KATs
def _ddim():
    return oddim.DDIMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear",
                               num_train_timesteps=1000, clip_sample=False)


def test_ddim_known_answers():
    s = _ddim()
    acp = s.alphas_cumprod
    assert abs(acp[0].item() - 0.99915) < 1e-6
    assert abs(acp[980].item() - 0.0058438) < 2e-7
    assert abs(acp[999].item() - 0.0046601) < 2e-7
    s.set_timesteps(50)
    assert s.timesteps.tolist() == list(range(980, -1, -20))
    s.set_timesteps(1000)
    for k in (1, 7, 49):
        assert int(s.timesteps[20 * k]) == 999 - 20 * k  # train_lora_xl.py:229-233
    assert s.init_noise_sigma == 1.0


def test_ddim_step_algebra():
    s = _ddim()
    s.set_timesteps(50)
    g = torch.Generator().manual_seed(0)
    x, eps = torch.randn(2, 4, 8, 8, generator=g), torch.randn(2, 4, 8, 8, generator=g)
    t = 500
    prev = s.step(eps, t, x).prev_sample
    a_t, a_p = s.alphas_cumprod[t], s.alphas_cumprod[t - 20]
    x0 = (x - (1 - a_t).sqrt() * eps) / a_t.sqrt()
    assert torch.allclose(prev, a_p.sqrt() * x0 + (1 - a_p).sqrt() * eps, atol=1e-6)
    # last step uses final_alpha_cumprod = 1: x_prev == predicted x0
    last = s.step(eps, 0, x).prev_sample
    a0 = s.alphas_cumprod[0]
    assert torch.allclose(last, (x - (1 - a0).sqrt() * eps) / a0.sqrt(), atol=1e-6)
    # add_noise / step round trip: stepping from t to t-20 with the true noise lands on the t-20 noising of x0
    x0 = torch.randn(2, 4, 8, 8, generator=g)
    xt = s.add_noise(x0, eps, torch.tensor([t]))
    back = s.step(eps, t, xt).prev_sample
    assert torch.allclose(back, s.add_noise(x0, eps, torch.tensor([t - 20])), atol=1e-5)


# ---------------------------------------------------------------------------------------- oracle numerics
def _tiny(cfg_name="tiny_xl", seed=11, dtype=torch.float32):
    m = ounet.UNet2DConditionModel(getattr(ounet.UNetConfig, cfg_name)())
    synthetic.init_synthetic_(m, seed=seed)
    return m.to(dtype).eval()


def test_fp32_vs_fp64_self_consistency():
    m32 = _tiny()
    m64 = _tiny(dtype=torch.float64)
    g = torch.Generator().manual_seed(3)
    x = torch.randn(1, 4, 16, 16, generator=g)
    ehs = torch.randn(1, 77, 256, generator=g)
    added = {"text_embeds": torch.randn(1, 128, generator=g), "time_ids": torch.tensor([[128., 128, 0, 0, 128, 128]])}
    with torch.no_grad():
        a = m32(x, 321, ehs, added_cond_kwargs=added).sample
        b = m64(x.double(), 321, ehs.double(),
                added_cond_kwargs={k: v.double() for k, v in added.items()}).sample
    rel = ((a.double() - b).norm() / b.norm()).item()
    assert rel < 1e-5, rel
    assert 0.1 < b.std().item() < 10  # synthetic weights keep activations O(1)


def test_oracle_matches_golden_no_lora():
    """Golden eps were produced by the reference's predict_noise_xl on this oracle; re-deriving the guided eps
    here (no reference code) must reproduce them bit-for-bit-ish (same torch, same seed-derived weights)."""
    fx = torch.load(os.path.join(GOLDEN, "tiny_xl.pt"))
    m = _tiny("tiny_xl", seed=fx["weight_seed"])
    with torch.no_grad():
        out = m(torch.cat([fx["latents"]] * 2), fx["timestep"], fx["text_embeddings"],
                added_cond_kwargs={"text_embeds": fx["add_text_embeddings"], "time_ids": fx["add_time_ids"]}).sample
    u, c = out.chunk(2)
    assert torch.allclose(u + 1 * (c - u), fx["eps_off_g1"], atol=2e-5, rtol=1e-4)
    assert torch.allclose(u + 3 * (c - u), fx["eps_off_g3"], atol=5e-5, rtol=1e-4)


def _fold_lora(model, fx, slider):
    """W += slider * alpha/r * up @ down with the fixture's seeded LoRA weights — algebraically the hook."""
    from sliders_b200 import lora as plora
    from sliders_b200.unet import UNet2DConditionModel as PU, UNetConfig as PC

    with torch.device("meta"):
        shell = PU(PC.from_dict(getattr(ounet.UNetConfig, fx["config"])().__dict__))
    with c3lier(plora):
        net = plora.LoRANetwork(shell, rank=fx["rank"], multiplier=1.0, alpha=fx["alpha"], train_method="noxattn")
    net = net.to_empty(device="cpu")
    for l in net.unet_loras:  # to_empty drops the alpha buffer value
        l.alpha.fill_(fx["alpha"])
    synthetic.init_lora_nonzero_(net, seed=fx["lora_seed"], up_std=fx["up_std"], reseed_down=True)
    mods = {("lora_unet_" + n.replace(".", "_")): mm for n, mm in model.named_modules()}
    sd = net.state_dict()
    with torch.no_grad():
        for l in net.unet_loras:
            up, down = sd[l.lora_name + ".lora_up.weight"].float(), sd[l.lora_name + ".lora_down.weight"].float()
            delta = torch.einsum("or,rikl->oikl", up[:, :, 0, 0], down) if down.dim() == 4 else up @ down
            mods[l.lora_name].weight.add_(delta * (slider * l.scale))
    return len(net.unet_loras)


def test_oracle_with_folded_lora_matches_reference_hook_golden():
    """The GPU parity tests compare against the oracle with W + s*up@down folded weights.  This test pins that
    shortcut to the reference's real forward hook (golden eps_on_* came from lora.py:108-112 running live)."""
    fx = torch.load(os.path.join(GOLDEN, "tiny_xl.pt"))
    m = _tiny("tiny_xl", seed=fx["weight_seed"])
    n = _fold_lora(m, fx, slider=1.0)
    assert n == fx["n_lora"]
    with torch.no_grad():
        out = m(torch.cat([fx["latents"]] * 2), fx["timestep"], fx["text_embeddings"],
                added_cond_kwargs={"text_embeds": fx["add_text_embeddings"], "time_ids": fx["add_time_ids"]}).sample
    u, c = out.chunk(2)
    got = u + 1 * (c - u)
    rel = ((got - fx["eps_on_s1_g1"]).norm() / fx["eps_on_s1_g1"].norm()).item()
    assert rel < 1e-5, rel
    eff = ((fx["eps_on_s1_g1"] - fx["eps_off_g1"]).norm() / fx["eps_off_g1"].norm()).item()
    assert eff > 1e-2  # the adaptor really changes the prediction


def test_golden_loss_formula():
    fx = torch.load(os.path.join(GOLDEN, "tiny_xl.pt"))
    tgt, pos, neu, unc = fx["eps_on_s1_g1"], fx["eps_off_g3"], fx["eps_off_g1"], fx["eps_on_sm2_g3"]
    want = torch.nn.functional.mse_loss(tgt, neu + 4.0 * (pos - unc))  # prompt_util.py:123-135 (enhance)
    assert torch.allclose(want, fx["loss_enhance_g4"], rtol=1e-5)


# ---------------------------------------------------------------------------------------- reference LoRA interface
def test_zero_init_identity_and_multiplier_semantics_with_reference_lora():
    """Identity and multiplier semantics of the LoRA hook through predict_noise_xl, run by the CPU port of hook + call on
    the oracle UNet, and the port's outputs against those of the reference's own code on the same weights and inputs
    (golden, reference_calls.pt)."""
    fx = torch.load(os.path.join(GOLDEN, "reference_calls.pt"))["hook_xl"]
    m = _tiny("tiny_xl", seed=fx["weight_seed"])
    m.requires_grad_(False)
    g = torch.Generator().manual_seed(fx["input_seed"])
    lat = torch.randn(1, 4, 16, 16, generator=g)
    ehs = torch.randn(2, 77, 256, generator=g)
    pooled = torch.randn(2, 128, generator=g)
    tids = torch.tensor([[128., 128, 0, 0, 128, 128]] * 2)
    t = fx["timestep"]
    sched = _ddim()
    sched.set_timesteps(1000)

    def close(a, b):
        return ((a - b).norm() / b.norm()).item() < 1e-5

    with torch.no_grad():
        base = port.predict_noise_xl(m, sched, t, lat, ehs, pooled, tids, guidance_scale=1)
        assert close(base, fx["base"])
        net = port.LoRAHooks(m, rank=fx["rank"], alpha=fx["alpha"], c3lier=True)
        with net:  # fresh LoRA: lora_up == 0 -> identity (lora.py:97-98)
            fresh = port.predict_noise_xl(m, sched, t, lat, ehs, pooled, tids, guidance_scale=1)
        assert torch.equal(fresh, base)
        synthetic.init_lora_nonzero_(net, seed=fx["lora_seed"], up_std=fx["up_std"], reseed_down=True)
        off = port.predict_noise_xl(m, sched, t, lat, ehs, pooled, tids, guidance_scale=1)  # multiplier 0 after exit
        assert torch.allclose(off, base, atol=1e-6)
        with net:
            on = port.predict_noise_xl(m, sched, t, lat, ehs, pooled, tids, guidance_scale=1)
        assert (on - base).abs().max() > 1e-3
        assert close(on, fx["on"])
        # guidance_scale = 1 => guided == text half (train_util.py:250-253)
        out = m(torch.cat([lat] * 2), t, ehs, added_cond_kwargs={"text_embeds": pooled, "time_ids": tids}).sample
        assert torch.allclose(base, out.chunk(2)[1], atol=1e-6)


def test_reference_state_dict_keys_match_ours():
    from sliders_b200 import lora as plora
    from sliders_b200.unet import UNet2DConditionModel as PU, UNetConfig as PC

    ref_keys = _reference_lora_keys()["state_dict_keys"]
    for name, cfg_o, cfg_p in (("sdxl", ounet.UNetConfig.sdxl(), PC.sdxl()), ("sd15", ounet.UNetConfig.sd15(), PC.sd15())):
        with torch.device("meta"):
            mo, mp = ounet.UNet2DConditionModel(cfg_o), PU(cfg_p)
            assert list(mo.state_dict().keys()) == list(mp.state_dict().keys())
            assert [tuple(v.shape) for v in mo.state_dict().values()] == [tuple(v.shape) for v in mp.state_dict().values()]
            for method in ("noxattn", "full", "xattn", "selfattn", "innoxattn", "xattn-strict", "noxattn-hspace",
                           "noxattn-hspace-last"):
                with c3lier(plora):
                    b = plora.LoRANetwork(mp, rank=4, multiplier=1.0, alpha=1.0, train_method=method)
                assert list(b.state_dict().keys()) == ref_keys[f"{name}/{method}"], method
                # re-create a fresh model: injection swaps the leaf forwards
                mp = PU(cfg_p)


def test_euler_discrete_known_answers_and_ddim_equivalence():
    """oracle/euler.py: sigma known answers for the SD betas (sigma_max 14.6146, sigma_min 0.0292), the SDXL config's
    timestep grid (leading, offset 1: 981, 961, ..., 1 for 50 steps) and init_noise_sigma, and the exact
    correspondence with DDIM (eta 0): on a shared integer grid x_euler = sqrt(1 + sigma^2) * x_ddim at every step."""
    from oracle import ddim as oddim
    from oracle import euler as oeuler

    kw = dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", num_train_timesteps=1000)
    e = oeuler.EulerDiscreteScheduler(timestep_spacing="leading", steps_offset=1, **kw)
    assert abs(float(e.sigmas.max()) - 14.6146) < 1e-3 and abs(float(e.sigmas[-2]) - 0.0292) < 1e-4
    assert abs(float(e.init_noise_sigma) - (14.6146 ** 2 + 1) ** 0.5) < 1e-3
    e.set_timesteps(50)
    assert [float(t) for t in e.timesteps[:3]] == [981.0, 961.0, 941.0] and float(e.timesteps[-1]) == 1.0
    assert float(e.sigmas[-1]) == 0.0 and len(e.sigmas) == 51
    lin = oeuler.EulerDiscreteScheduler(timestep_spacing="linspace", **kw)
    assert abs(float(lin.init_noise_sigma) - 14.6146) < 1e-3
    # equivalence with DDIM on the same (integer, leading, offset 0) grid
    n = 20
    e0 = oeuler.EulerDiscreteScheduler(timestep_spacing="leading", steps_offset=0, **kw)
    e0.set_timesteps(n)
    d = oddim.DDIMScheduler(clip_sample=False, **kw)
    d.set_timesteps(n)
    assert [int(t) for t in d.timesteps] == [int(t) for t in e0.timesteps]
    g = torch.Generator().manual_seed(0)
    x_vp = torch.randn(1, 4, 8, 8, generator=g, dtype=torch.float64)
    x_ve = x_vp * (float(e0.sigmas[0]) ** 2 + 1) ** 0.5
    for i, t in enumerate(d.timesteps):
        eps = torch.randn(1, 4, 8, 8, generator=g, dtype=torch.float64)
        assert torch.allclose(e0.scale_model_input(x_ve, float(t)), x_vp, rtol=1e-4, atol=1e-5)
        x_vp = d.step(eps, int(t), x_vp).prev_sample
        x_ve = e0.step(eps, float(t), x_ve).prev_sample
        s_next = float(e0.sigmas[i + 1])
        assert torch.allclose(x_ve, x_vp * (s_next ** 2 + 1) ** 0.5, rtol=2e-4, atol=2e-4)


def test_lms_discrete_properties():
    """oracle/lms.py: first step == Euler step; coefficients sum to d sigma; a cubic-in-sigma derivative is integrated
    exactly from the fourth step on (order-4 Adams-Bashforth on a non-uniform grid)."""
    from oracle import euler as oeuler
    from oracle import lms as olms

    kw = dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", num_train_timesteps=1000)
    l = olms.LMSDiscreteScheduler(**kw)
    e = oeuler.EulerDiscreteScheduler(timestep_spacing="linspace", **kw)
    assert abs(float(l.init_noise_sigma) - 14.6146) < 1e-3
    l.set_timesteps(30)
    e.set_timesteps(30)
    assert torch.equal(l.timesteps, e.timesteps) and torch.equal(l.sigmas, e.sigmas)
    g = torch.Generator().manual_seed(0)
    x = torch.randn(1, 4, 8, 8, generator=g, dtype=torch.float64) * 14.6
    eps = torch.randn(1, 4, 8, 8, generator=g, dtype=torch.float64)
    t0 = float(l.timesteps[0])
    assert torch.allclose(l.step(eps, t0, x).prev_sample, e.step(eps, t0, x).prev_sample, rtol=1e-6, atol=1e-6)
    for i in (1, 2, 5, 20):
        order = min(i + 1, 4)
        cs = [l.get_lms_coefficient(order, i, k) for k in range(order)]
        assert abs(sum(cs) - float(l.sigmas[i + 1] - l.sigmas[i])) < 1e-4 * abs(float(l.sigmas[i]))
    # exactness for cubic derivatives: d(sigma) = a + b s + c s^2 + d s^3, x(s) = integral
    l.set_timesteps(30)
    a, b, c, d3 = 0.3, -0.2, 0.05, -0.004
    f = lambda s: a + b * s + c * s ** 2 + d3 * s ** 3
    F = lambda s: a * s + b * s ** 2 / 2 + c * s ** 3 / 3 + d3 * s ** 4 / 4
    x = torch.tensor([F(float(l.sigmas[0]))], dtype=torch.float64)
    for i, t in enumerate(l.timesteps[:8]):
        s = float(l.sigmas[i])
        eps = torch.tensor([f(s)], dtype=torch.float64)   # derivative == eps for epsilon prediction
        x_next = l.step(eps, float(t), x).prev_sample
        if i >= 3:
            assert abs(float(x_next) - F(float(l.sigmas[i + 1]))) < 2e-3, i
        x = torch.tensor([F(float(l.sigmas[i + 1]))], dtype=torch.float64)  # restart from the exact value


def test_stochastic_sampler_identities():
    """oracle/stochastic.py (DDPM / Euler-ancestral restatements) against closed forms that do not depend on the
    restatement: the DDPM posterior q(x_{t-1} | x_t, x_0) and the ancestral variance split."""
    from oracle import stochastic as ost

    kw = dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear")
    d = ost.DDPMScheduler(clip_sample=False, **kw)
    d.set_timesteps(1000)
    acp = d.alphas_cumprod.double()
    g = torch.Generator().manual_seed(0)
    x0 = torch.randn(1, 4, 8, 8, generator=g).double()
    eps = torch.randn(1, 4, 8, 8, generator=g).double()
    for t in (999, 500, 37, 1):
        xt = d.add_noise(x0, eps, torch.tensor([t]))
        # with the TRUE eps the predicted x0 is exact, so the step's mean is the posterior mean of Ho et al. eq. 7
        zeros = torch.Generator().manual_seed(1)
        out = d.step(eps, t, xt, generator=zeros)
        assert torch.allclose(out.pred_original_sample, x0, atol=1e-5)
        beta_t = 1 - acp[t] / acp[t - 1]
        mean = (acp[t - 1].sqrt() * beta_t / (1 - acp[t])) * x0 + ((acp[t] / acp[t - 1]).sqrt() * (1 - acp[t - 1]) / (1 - acp[t])) * xt
        var = (1 - acp[t - 1]) / (1 - acp[t]) * beta_t
        z = torch.randn(xt.shape, generator=torch.Generator().manual_seed(1), dtype=torch.float64)
        assert torch.allclose(out.prev_sample, mean + var.sqrt() * z, atol=1e-5)
    # t = 0: no noise, the step returns x0 itself
    xt = d.add_noise(x0, eps, torch.tensor([0]))
    assert torch.allclose(d.step(eps, 0, xt).prev_sample, x0, atol=1e-5)

    e = ost.EulerAncestralDiscreteScheduler(**kw)
    e.set_timesteps(30)
    s = e.sigmas.double()
    assert abs(float(e.init_noise_sigma) - 14.6146) < 1e-3 and float(s[-1]) == 0.0
    for i in range(30):
        up2 = s[i + 1] ** 2 * (s[i] ** 2 - s[i + 1] ** 2) / s[i] ** 2
        down2 = s[i + 1] ** 2 - up2
        assert up2 >= 0 and down2 >= -1e-12 and abs(float(up2 + down2 - s[i + 1] ** 2)) < 1e-9
    # noise-free part == an Euler step to sigma_down; last step (sigma_to = 0) is deterministic and returns x - sigma eps
    x = torch.randn(1, 4, 8, 8, generator=g).double() * float(s[0])
    t_last = e.timesteps[-1]
    assert torch.allclose(e.step(eps, t_last, x).prev_sample, x - s[-2] * eps, atol=1e-6)


def test_port_reproduces_the_reference_loop_golden():
    """oracle/port.py (the CPU port bench.py falls back to where /root/reference is absent) against the fixture the
    reference's own loop source produced (tests/golden/iter_text_xl.pt): same adaptor set, same loss, same gradients."""
    import os

    from oracle import port
    from sliders_b200 import synthetic

    fx = torch.load(os.path.join(os.path.dirname(__file__), "golden", "iter_text_xl.pt"))
    cfg = ounet.UNetConfig.tiny_xl()
    om = ounet.UNet2DConditionModel(cfg)
    synthetic.init_synthetic_(om, seed=fx["weight_seed"])
    om.requires_grad_(False).eval()
    net = port.LoRAHooks(om, rank=fx["rank"], alpha=fx["alpha"], c3lier=True)
    assert len(net.unet_loras) == fx["n_lora"]
    assert {k for k, _ in net.named_parameters()} == set(fx["grads"])
    synthetic.init_lora_nonzero_(net, seed=fx["lora_seed"], up_std=fx["up_std"], reseed_down=True)
    net.__exit__()
    sched = oddim.DDIMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear",
                                num_train_timesteps=1000, clip_sample=False)
    opt = torch.optim.AdamW(net.prepare_optimizer_params(), lr=fx["lr"])
    emb = {k: v[0] for k, v in fx["embeds"].items()}
    added = {k: (v[1], fx["add_time_ids"]) for k, v in fx["embeds"].items()}
    loss = port.text_slider_iteration(om, net, sched, opt, emb, fx["latents"], fx["timesteps_to"],
                                      guidance_scale=fx["settings"]["guidance_scale"], action=fx["settings"]["action"],
                                      added=added)
    assert abs(float(loss) - float(fx["loss"])) < 1e-5 * max(1.0, abs(float(fx["loss"])))
    num = den = 0.0
    for k, p in net.named_parameters():
        # (the optimizer step ran after backward; .grad is untouched by it)
        num += (p.grad - fx["grads"][k].float()).pow(2).sum().item()
        den += fx["grads"][k].float().pow(2).sum().item()
    assert (num / den) ** 0.5 < 5e-3   # the fixture stores bf16-rounded gradients
