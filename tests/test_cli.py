"""CPU tests of the trainers' command line (sliders_b200/cli.py, config_util.py, prompt_util.py, model_util.py): the YAML
schema and the flag semantics of the reference's train_lora*.py, checked against what the reference's own config_util /
prompt_util modules make of the reference's data files (tests/golden/make_golden_reference.py)."""
import os
import sys

import pytest
import torch

from sliders_b200 import cli, config_util, model_util, prompt_util

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DATA = os.path.join(ROOT, "trainscripts", "textsliders", "data")
GOLDEN = os.path.join(ROOT, "tests", "golden")
REF_DATA = os.path.join(GOLDEN, "reference_data")   # the reference's own data files, verbatim


def test_shipped_yaml_parses_and_builds_pairs():
    cfg = config_util.load_config_from_yaml(os.path.join(DATA, "config-xl.yaml"))
    assert (cfg.network.type, cfg.network.rank, cfg.network.training_method) == ("c3lier", 4, "noxattn")
    assert cfg.train.noise_scheduler == "ddim" and cfg.train.max_denoising_steps == 50
    assert config_util.parse_precision(cfg.train.precision) is torch.bfloat16
    with pytest.raises(ValueError):
        config_util.parse_precision("int8")
    prompts = prompt_util.load_prompts_from_yaml(os.path.join(ROOT, cfg.prompts_file), ["male", "female"])
    assert [p.target for p in prompts] == ["male person", "female person"]
    assert prompts[0].positive == "male person, smiling broadly" and prompts[0].action == "enhance"
    pairs = cli.build_prompt_pairs(prompts, True, "cpu", torch.float32, synthetic=True)
    assert len(pairs) == 2 and pairs[0].target.text_embeds.shape == (1, 77, 2048)
    assert pairs[0].target.pooled_embeds.shape == (1, 1280) and pairs[0].guidance_scale == 4
    # the cache hands the same object to identical prompt strings (target == neutral here)
    assert pairs[0].target is pairs[0].neutral and pairs[0].target is not pairs[1].target
    sd = cli.build_prompt_pairs(prompts, False, "cpu", torch.float32, synthetic=True)
    assert sd[0].positive.shape == (1, 77, 768)
    with pytest.raises(KeyError, match="no embedding for prompt"):
        cli.build_prompt_pairs(prompts, True, "cpu", torch.float32)


def test_prompt_defaults_and_unknown_keys():
    s = prompt_util.PromptSettings(target="van gogh", guidance=3, rank=4)       # GPT-written files carry extra keys
    assert (s.positive, s.unconditional, s.neutral, s.action, s.resolution) == ("van gogh", "", "", "erase", 512)
    with pytest.raises(Exception):
        prompt_util.PromptSettings(positive="x")
    cache = prompt_util.PromptEmbedsCache()
    assert cache["a"] is None
    cache["a"] = 1
    assert cache["a"] == 1


def test_flag_overrides_and_save_cadence(tmp_path):
    cfg = config_util.load_config_from_yaml(os.path.join(DATA, "config-xl.yaml"))
    args = cli.build_parser("text_xl").parse_args(["--config_file", "x", "--name", "ageslider", "--rank", "8", "--alpha",
                                                   "2", "--attributes", "male, female", "--prompts_file", "p.yaml"])
    cfg = cli.apply_overrides(cfg, args, "text_xl")
    assert cfg.save.name == "ageslider_alpha2.0_rank8_noxattn" and cfg.save.path == "./models/ageslider_alpha2.0_rank8_noxattn"
    assert cfg.prompts_file == "p.yaml" and cli.split_csv(args.attributes) == ["male", "female"]
    cfg.train.iterations, cfg.save.per_steps = 1001, 500
    assert [i for i in range(1001) if cli.should_save(i, cfg)] == [500]        # not 0, not the last iteration
    # image sliders: --alpha required, rank defaults to 4, folders / scales lists
    with pytest.raises(SystemExit):
        cli.build_parser("image_xl").parse_args(["--config_file", "x", "--folder_main", "d"])
    ia = cli.build_parser("image_xl").parse_args(["--config_file", "x", "--folder_main", "d", "--alpha", "1"])
    assert ia.rank == 4 and cli.split_csv(ia.folders) == ["verylow", "low", "high", "veryhigh"]
    assert [int(s) for s in cli.split_csv(ia.scales)] == [-2, -1, 1, 2]
    # latent folders
    (tmp_path / "low").mkdir()
    (tmp_path / "low" / "a.png").write_bytes(b"")
    with pytest.raises(FileNotFoundError, match="encode them with the SD VAE"):
        cli.list_pairs(str(tmp_path), "low", "high")
    torch.save(torch.zeros(4, 8, 8), tmp_path / "low" / "a.pt")
    assert cli.list_pairs(str(tmp_path), "low", "high") == ["a.pt"]
    assert cli.load_latent(str(tmp_path / "low" / "a.pt")).shape == (1, 4, 8, 8)


def test_model_sources():
    with pytest.raises(FileNotFoundError, match="never downloads"):
        model_util._resolve("stabilityai/definitely-not-cached")
    assert model_util._resolve("synthetic:7") == ("synthetic", "synthetic:7")
    with pytest.raises(ValueError):
        model_util.create_noise_scheduler("plms")
    for name in model_util.AVAILABLE_SCHEDULERS:        # every name the reference's factory accepts
        assert model_util.create_noise_scheduler(name) is not None


def test_reference_yaml_files_parse_like_the_reference():
    ref = torch.load(os.path.join(GOLDEN, "reference_calls.pt"))["yaml"]   # the reference parsers' `.dict()`
    for name in ("config-xl.yaml", "config.yaml"):
        ours = config_util.load_config_from_yaml(os.path.join(REF_DATA, name))
        assert ours.model_dump() == ref[name]
    for name, atts in (("prompts-xl.yaml", ["male", "female"]), ("prompts.yaml", []),
                       ("prompts-person_age_slider_GPT.yaml", ["asian", "white"])):
        ours = prompt_util.load_prompts_from_yaml(os.path.join(REF_DATA, name), atts)
        assert len(ref[name]) > 0 and [o.model_dump() for o in ours] == ref[name]


def test_eval_sweep_host_logic(tmp_path):
    """eval-scripts/generate_images_xl.py:445-508 driver pieces: CSV rows, slider-name parsing, seeded start noise."""
    from sliders_b200 import eval_sweep as es

    rows = es.read_prompts_csv(os.path.join(ROOT, "prompts", "prompts-sample.csv"), from_case=1)
    assert [r["case_number"] for r in rows] == [1, 2] and rows[0]["seed"] == 54737 and rows[1]["prompt"].startswith("photo")
    info = es.parse_slider_name("models/ageslider_alpha1.0_rank4_noxattn/ageslider_alpha1.0_rank4_noxattn_last.pt")
    assert (info["rank"], info["alpha"], info["train_method"], info["network_type"]) == (4, 1.0, "noxattn", "c3lier")
    assert es.parse_slider_name("x_rank8_full.pt")["train_method"] == "full" and es.parse_slider_name("x.pt")["rank"] == 1
    a = es.initial_latents(7, 2, 64, 64, 2.0, "cpu", torch.float32)
    torch.manual_seed(7)
    assert torch.equal(a, torch.randn(2, 4, 8, 8) * 2.0)      # == generator = torch.manual_seed(seed) + prepare_latents
    args = es.build_parser().parse_args(["--model_name", "m.pt", "--prompts_path", "p.csv", "--save_path", "o"])
    assert (args.start_noise, args.rank, args.num_samples, args.ddim_steps) == (750, 4, 1, 50)
    ref = es.read_prompts_csv(os.path.join(REF_DATA, "prompts-person.csv"))   # the reference's own prompt file
    assert len(ref) > 10 and ref[0]["prompt"] == "image of a person"
