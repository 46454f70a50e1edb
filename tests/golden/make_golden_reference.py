"""Generates the fixtures that stand in for the reference tree in the CPU tests — run where the reference's sources are
available (`SLIDERS_REFERENCE_ROOT`, see oracle/reference_bridge.py):

    python tests/golden/make_golden_reference.py

What the tests used to ask the reference's own, unmodified modules at run time is recorded here once:
  * reference_lora_keys.json.gz — `LoRANetwork` (lora.py) on the oracle UNet: the state-dict keys of every
    `train_method` for SDXL and SD1.x (c3lier leaf set), the adaptor / parameter counts of the shipped configurations,
    and the key -> shape table of the small UNet the checkpoint round-trip test writes;
  * reference_calls.pt — `predict_noise_xl` (train_util.py) with the LoRA hook fresh / off / on on the tiny SDXL oracle,
    `PromptEmbedsPair.loss` (prompt_util.py) for both actions, and the parsed form (`.dict()`) of the reference's YAML
    files under config_util / prompt_util;
  * reference_data/ — those YAML files and the evaluation prompt CSV, verbatim (data fixtures, inputs of the parsers).
"""
import gzip
import json
import os
import shutil
import sys

import torch

OUT = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(OUT))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from conftest import c3lier  # noqa: E402
from oracle import reference_bridge as rb  # noqa: E402
from oracle import unet as ounet  # noqa: E402
from sliders_b200 import synthetic  # noqa: E402

METHODS = ("noxattn", "full", "xattn", "selfattn", "innoxattn", "xattn-strict", "noxattn-hspace", "noxattn-hspace-last")
YAML_FILES = (("config-xl.yaml", None), ("config.yaml", None), ("prompts-xl.yaml", ["male", "female"]),
              ("prompts.yaml", []), ("prompts-person_age_slider_GPT.yaml", ["asian", "white"]))
CSV_FILE = "prompts-person.csv"
# the small two-level UNet of tests/test_host.py::test_checkpoint_roundtrip_pt_and_safetensors
SMALL_UNET = dict(block_out_channels=(64, 128), down_block_types=("DownBlock2D", "CrossAttnDownBlock2D"),
                  up_block_types=("CrossAttnUpBlock2D", "UpBlock2D"), transformer_layers_per_block=(1, 1),
                  attention_head_dim=(1, 2), cross_attention_dim=64)


def lora_keys(lora):
    keys, counts = {}, {}
    for cfg_name in ("sdxl", "sd15"):
        for method in METHODS:
            with torch.device("meta"):
                m = ounet.UNet2DConditionModel(getattr(ounet.UNetConfig, cfg_name)())
                with c3lier(lora):
                    net = lora.LoRANetwork(m, rank=4, multiplier=1.0, alpha=1.0, train_method=method)
            keys[f"{cfg_name}/{method}"] = list(net.state_dict().keys())
    for cfg_name, rank in (("sdxl", 4), ("sdxl", 8), ("sd15", 4)):
        with torch.device("meta"):
            m = ounet.UNet2DConditionModel(getattr(ounet.UNetConfig, cfg_name)())
            with c3lier(lora):
                net = lora.LoRANetwork(m, rank=rank, multiplier=1.0, alpha=1.0, train_method="noxattn")
        counts[f"{cfg_name}/{rank}"] = {"n_leaves": len(net.unet_loras),
                                        "n_params": sum(p.numel() for p in net.parameters()),
                                        "lora_names": [l.lora_name for l in net.unet_loras]}
    om = ounet.UNet2DConditionModel(ounet.UNetConfig(**SMALL_UNET))
    with c3lier(lora):
        net = lora.LoRANetwork(om, rank=4, multiplier=1.0, alpha=1.0, train_method="noxattn")
    small = {k: list(v.shape) for k, v in net.state_dict().items()}
    return {"state_dict_keys": keys, "counts": counts, "small_unet_checkpoint": small}


def hook_calls(lora, tu, mu):
    """The fresh / off / on behaviour of the LoRA hook through the reference's predict_noise_xl (tiny SDXL oracle)."""
    m = ounet.UNet2DConditionModel(ounet.UNetConfig.tiny_xl())
    synthetic.init_synthetic_(m, seed=11)
    m.eval().requires_grad_(False)
    g = torch.Generator().manual_seed(5)
    lat = torch.randn(1, 4, 16, 16, generator=g)
    ehs = torch.randn(2, 77, 256, generator=g)
    pooled = torch.randn(2, 128, generator=g)
    tids = torch.tensor([[128., 128, 0, 0, 128, 128]] * 2)
    sched = mu.create_noise_scheduler("ddim")
    sched.set_timesteps(1000)
    # inputs are not stored: the test redraws them from the same seed
    fx = {"weight_seed": 11, "lora_seed": 1, "up_std": 0.05, "rank": 4, "alpha": 1.0, "timestep": 500, "input_seed": 5}
    with torch.no_grad():
        fx["base"] = tu.predict_noise_xl(m, sched, 500, lat, ehs, pooled, tids, guidance_scale=1)
        with c3lier(lora):
            net = lora.LoRANetwork(m, rank=4, multiplier=1.0, alpha=1.0, train_method="noxattn")
        with net:  # fresh LoRA: lora_up == 0 (lora.py:97-98)
            fx["fresh"] = tu.predict_noise_xl(m, sched, 500, lat, ehs, pooled, tids, guidance_scale=1)
        synthetic.init_lora_nonzero_(net, seed=1, up_std=0.05, reseed_down=True)
        fx["off"] = tu.predict_noise_xl(m, sched, 500, lat, ehs, pooled, tids, guidance_scale=1)  # multiplier 0
        with net:
            fx["on"] = tu.predict_noise_xl(m, sched, 500, lat, ehs, pooled, tids, guidance_scale=1)
        out = m(torch.cat([lat] * 2), 500, ehs, added_cond_kwargs={"text_embeds": pooled, "time_ids": tids}).sample
        fx["text_half"] = out.chunk(2)[1].clone()
    # sanity of the recorded run (the test checks the same properties on the port)
    assert torch.equal(fx["fresh"], fx["base"]) and torch.allclose(fx["off"], fx["base"], atol=1e-6)
    assert (fx["on"] - fx["base"]).abs().max() > 1e-3 and torch.allclose(fx["base"], fx["text_half"], atol=1e-6)
    return fx


def prompt_pair_losses(pu):
    g = torch.Generator().manual_seed(1)
    t, p, u, n = (torch.randn(2, 4, 8, 8, generator=g) for _ in range(4))
    fx = {"target": t, "positive": p, "unconditional": u, "neutral": n, "guidance_scale": 2.5, "batch_size": 2}
    for action in ("erase", "enhance"):
        rs = pu.PromptSettings(target="t", positive="p", unconditional="u", neutral="n", action=action,
                               guidance_scale=2.5, resolution=512, batch_size=2)
        ref = pu.PromptEmbedsPair(torch.nn.MSELoss(), None, None, None, None, rs)
        fx[action] = {"loss": ref.loss(target_latents=t, positive_latents=p, unconditional_latents=u, neutral_latents=n),
                      "batch_size": ref.batch_size, "resolution": ref.resolution, "dynamic_crops": ref.dynamic_crops}
    return fx


def main():
    assert rb.available(), f"needs the reference tree at {rb.REFERENCE_ROOT} (set SLIDERS_REFERENCE_ROOT)"
    lora, tu, mu = rb.load("lora"), rb.load("train_util"), rb.load("model_util")
    rc, pu = rb.load("config_util"), rb.load("prompt_util")

    with open(os.path.join(OUT, "reference_lora_keys.json.gz"), "wb") as f:
        f.write(gzip.compress(json.dumps(lora_keys(lora)).encode(), mtime=0))

    data = os.path.join(OUT, "reference_data")
    os.makedirs(data, exist_ok=True)
    src = os.path.join(rb.REFERENCE_ROOT, "trainscripts", "textsliders", "data")
    parsed = {}
    for name, atts in YAML_FILES:
        shutil.copyfile(os.path.join(src, name), os.path.join(data, name))
        if atts is None:
            parsed[name] = rc.load_config_from_yaml(os.path.join(data, name)).dict()
        else:
            parsed[name] = [r.dict() for r in pu.load_prompts_from_yaml(os.path.join(data, name), atts)]
    shutil.copyfile(os.path.join(rb.REFERENCE_ROOT, "prompts", CSV_FILE), os.path.join(data, CSV_FILE))

    fx = {"hook_xl": hook_calls(lora, tu, mu), "prompt_pair": prompt_pair_losses(pu), "yaml": parsed}
    torch.save(fx, os.path.join(OUT, "reference_calls.pt"))
    print({k: os.path.getsize(os.path.join(OUT, k)) for k in ("reference_lora_keys.json.gz", "reference_calls.pt")})


if __name__ == "__main__":
    main()
