"""CPU tests of the host-side logic: the C-ABI library loads and exports every declared symbol, the product
module tree / LoRANetwork mirror the reference interface, the product DDIM scheduler agrees with the oracle
restatement, checkpoints round-trip in the reference layout, and the multi-rank fan-out helpers reproduce the
single-rank result under gloo with world_size 2.  No GPU compute happens here."""
import gzip
import json
import os
import re
import subprocess
import sys

import pytest
import torch

from conftest import c3lier
from oracle import ddim as oddim
from sliders_b200 import _cabi, lora as plora, parallel, scheduler as psched, synthetic
from sliders_b200.unet import UNet2DConditionModel, UNetConfig

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


# ---------------------------------------------------------------------------------------- C ABI
def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "sb200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(sb200_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    import __graft_entry__ as ge

    if not os.path.exists(_cabi.lib_path()):
        ge.build()
    lib = _cabi.load()
    declared = _declared_symbols()
    assert len(declared) >= 15
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/sb200.h but not exported"
        assert name in _cabi.SIGNATURES, f"{name} has no ctypes prototype in _cabi.SIGNATURES"
    assert lib.sb200_version().decode() == "sb200 0.1 sm_100a"


def test_sass_contains_blackwell_tensor_and_tma_instructions():
    """`tcgen05.mma` shows up as UTC*MMA, TMA as UTMALDG, tcgen05.ld as LDTM (B200_PROFILING.md)."""
    if not os.path.exists(_cabi.lib_path()):
        pytest.skip("library not built")
    sass = subprocess.run(["cuobjdump", "-sass", _cabi.lib_path()], capture_output=True, text=True).stdout
    assert "UTCHMMA" in sass or "UTCMMA" in sass
    assert "UTMALDG" in sass
    assert "LDTM" in sass and "STTM" in sass
    assert "HMMA.16816" not in sass  # no legacy mma.sync path


def test_no_cpu_fallback():
    m = UNet2DConditionModel(UNetConfig.from_dict(dict(block_out_channels=(64, 128), down_block_types=(
        "DownBlock2D", "CrossAttnDownBlock2D"), up_block_types=("CrossAttnUpBlock2D", "UpBlock2D"),
        transformer_layers_per_block=(1, 1), attention_head_dim=(1, 2), cross_attention_dim=64)))
    with pytest.raises(RuntimeError, match="no CPU path"):
        m(torch.zeros(1, 4, 8, 8), 10, encoder_hidden_states=torch.zeros(1, 77, 64))
    with pytest.raises(RuntimeError, match="parameter container"):
        m.mid_block(torch.zeros(1))


# ---------------------------------------------------------------------------------------- module tree / LoRA API
@pytest.mark.parametrize("cfg,n_leaves,n_params", [(UNetConfig.sdxl(), 346, 4_320_000), (UNetConfig.sd15(), 150, 2_906_880)])
def test_product_lora_counts(cfg, n_leaves, n_params):
    with torch.device("meta"):
        m = UNet2DConditionModel(cfg)
        with c3lier(plora):
            net = plora.LoRANetwork(m, rank=4, multiplier=1.0, alpha=1.0, train_method="noxattn")
    assert len(net.unet_loras) == n_leaves
    assert sum(p.numel() for p in net.parameters()) == n_params
    # without c3lier only the Attention leaves (lierla)
    with torch.device("meta"):
        m = UNet2DConditionModel(cfg)
        net2 = plora.LoRANetwork(m, rank=4, alpha=1.0, train_method="noxattn")
    assert len(net2.unet_loras) == (280 if n_leaves == 346 else 64)


def test_lora_module_semantics():
    with torch.device("meta"):
        m = UNet2DConditionModel(UNetConfig.sd15())
    with c3lier(plora):
        net = plora.LoRANetwork(m, rank=8, multiplier=1.0, alpha=4.0, train_method="full")
    l = net.unet_loras[0]
    assert l.scale == 4.0 / 8 and l.lora_dim == 8 and float(l.alpha) == 4.0
    assert set(k.split(".", 1)[1] for k in net.state_dict() if k.startswith(l.lora_name + ".")) == {
        "alpha", "lora_down.weight", "lora_up.weight"}
    # context-manager semantics (lora.py:249-258)
    assert all(x.multiplier == 1.0 for x in net.unet_loras)  # constructor value before the first exit
    net.set_lora_slider(-3.0)
    with net:
        assert all(x.multiplier == -3.0 for x in net.unet_loras)
    assert all(x.multiplier == 0 for x in net.unet_loras)
    # the leaf's forward is swapped for the adaptor's bound method: how the engine discovers adaptors
    from sliders_b200.unet import _adaptor_of

    leaf = m.down_blocks[0].attentions[0].transformer_blocks[0].attn1.to_q
    assert _adaptor_of(leaf) is getattr(net, "lora_unet_down_blocks_0_attentions_0_transformer_blocks_0_attn1_to_q")
    with pytest.raises(RuntimeError, match="no eager path"):
        leaf.forward(torch.zeros(1))
    groups = net.prepare_optimizer_params()
    assert len(groups) == 1 and len(groups[0]["params"]) == 2 * len(net.unet_loras)
    conv = [x for x in net.unet_loras if x.lora_name.endswith("resnets_0_conv1")][0]
    assert conv.lora_down.weight.shape[2:] == (3, 3) and conv.lora_up.weight.shape[2:] == (1, 1)


def test_checkpoint_roundtrip_pt_and_safetensors(tmp_path):
    cfg = UNetConfig.from_dict(dict(block_out_channels=(64, 128), down_block_types=("DownBlock2D", "CrossAttnDownBlock2D"),
                                    up_block_types=("CrossAttnUpBlock2D", "UpBlock2D"),
                                    transformer_layers_per_block=(1, 1), attention_head_dim=(1, 2), cross_attention_dim=64))
    m = UNet2DConditionModel(cfg)
    with c3lier(plora):
        net = plora.LoRANetwork(m, rank=4, multiplier=1.0, alpha=1.0, train_method="noxattn")
    synthetic.init_lora_nonzero_(net, seed=3)
    for ext in (".pt", ".safetensors"):
        f = str(tmp_path / f"slider_alpha1.0_rank4_noxattn_last{ext}")
        net.save_weights(f, dtype=torch.bfloat16)
        if ext == ".pt":
            sd = torch.load(f)
        else:
            from safetensors.torch import load_file

            sd = load_file(f)
        assert all(v.dtype == torch.bfloat16 for v in sd.values())
        m2 = UNet2DConditionModel(cfg)
        with c3lier(plora):
            net2 = plora.LoRANetwork(m2, rank=4, multiplier=1.0, alpha=1.0, train_method="noxattn")
        missing = net2.load_state_dict(sd, strict=True)
        assert not missing.missing_keys and not missing.unexpected_keys
        for k, v in net.state_dict().items():
            assert torch.equal(net2.state_dict()[k].to(torch.bfloat16), v.to(torch.bfloat16)), k
    # a slider written by us loads strictly into the reference's own LoRANetwork on the oracle UNet: exactly its keys,
    # each with its shape (tests/golden/make_golden_reference.py records them)
    with gzip.open(os.path.join(GOLDEN, "reference_lora_keys.json.gz"), "rt") as f:
        ref = json.load(f)["small_unet_checkpoint"]
    sd = torch.load(str(tmp_path / "slider_alpha1.0_rank4_noxattn_last.pt"))
    assert {k: list(v.shape) for k, v in sd.items()} == ref


# ---------------------------------------------------------------------------------------- scheduler
def test_product_ddim_matches_oracle_ddim():
    a = psched.create_noise_scheduler("ddim")
    b = oddim.DDIMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear",
                            num_train_timesteps=1000, clip_sample=False)
    assert torch.equal(a.alphas_cumprod, b.alphas_cumprod)
    for n in (50, 1000, 30):
        a.set_timesteps(n)
        b.set_timesteps(n)
        assert torch.equal(a.timesteps, b.timesteps)
    a.set_timesteps(50)
    b.set_timesteps(50)
    g = torch.Generator().manual_seed(0)
    x, e = torch.randn(2, 4, 8, 8, generator=g), torch.randn(2, 4, 8, 8, generator=g)
    for t in (980, 500, 0):
        assert torch.allclose(a.step(e, t, x).prev_sample, b.step(e, t, x).prev_sample, atol=1e-6)
    ts = torch.tensor([300])
    assert torch.allclose(a.add_noise(x, e, ts), b.add_noise(x, e, ts))
    assert a.init_noise_sigma == 1.0 and a.scale_model_input(x, 3) is x
    with pytest.raises(ValueError):        # model_util.py:276-277: unknown names raise ValueError
        psched.create_noise_scheduler("dpm++")


# ---------------------------------------------------------------------------------------- multi-rank fan-out (gloo)
def test_shard_range_partitions():
    for n in (1, 3, 8, 11):
        for w in (1, 2, 4, 8):
            spans = [parallel.shard_range(n, r, w) for r in range(w)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(spans[i][1] == spans[i + 1][0] for i in range(w - 1))
            assert max(h - l for l, h in spans) - min(h - l for l, h in spans) <= 1


_WORKER = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from sliders_b200 import parallel
dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{sys.argv[2]}", rank=int(sys.argv[3]), world_size=2)
g = torch.Generator().manual_seed(0)
lat = torch.randn(5, 4, 8, 8, generator=g); emb = torch.randn(5, 7, 16, generator=g)
W = torch.randn(16, 4, generator=g)
def predict(l, e, scale=1.0):   # stand-in for the UNet: any per-pass-independent function
    return torch.tanh(l * scale) + (e.mean(1) @ W)[:, :, None, None]
full = predict(lat, emb, scale=0.5)
got = parallel.fanout_predict(predict, (lat, emb), scale=0.5)
assert torch.equal(got, full), "fan-out result differs from the single-rank result"
p = torch.nn.Parameter(torch.ones(6)); q = torch.nn.Parameter(torch.ones(2, 3))
if dist.get_rank() == 0:
    p.grad = torch.arange(6.0); q.grad = None          # rank 1 holds no graph for q... and rank 0 none for q
else:
    p.grad = torch.ones(6); q.grad = torch.full((2, 3), 2.0)
parallel.allreduce_lora_grads([p, q])
assert torch.equal(p.grad, torch.arange(6.0) + 1) and torch.equal(q.grad, torch.full((2, 3), 2.0))
dist.destroy_process_group()
print("ok")
'''


def test_fanout_two_ranks_gloo(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    port = 29500 + (os.getpid() % 2000)
    procs = [subprocess.Popen([sys.executable, str(script), ROOT, str(port), str(r)], stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=180)[0] for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0 and "ok" in o, o


_GROUPS_WORKER = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from sliders_b200 import parallel
dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{sys.argv[2]}", rank=int(sys.argv[3]), world_size=4)
rank = dist.get_rank()
grp, idx, n = parallel.slider_groups(2)
assert n == 2 and idx == rank // 2 and dist.get_world_size(grp) == 2
# each group is its own job: draws follow the group's rank 0, gradients are summed inside the group only
vals = parallel.sync_draws([float(rank), 7.0], "cpu", grp)
assert vals == [float(2 * idx), 7.0], vals
p = torch.nn.Parameter(torch.zeros(3)); p.grad = torch.full((3,), float(rank + 1))
parallel.allreduce_lora_grads([p], group=grp)
assert torch.equal(p.grad, torch.full((3,), float(4 * idx + 3))), p.grad    # (1+2) or (3+4)
net = torch.nn.Linear(2, 2); torch.nn.init.constant_(net.weight, float(rank)); torch.nn.init.zeros_(net.bias)
parallel.broadcast_lora_params(net, grp)
assert torch.equal(net.weight, torch.full((2, 2), float(2 * idx)))
parallel.assert_replicas_equal(list(net.parameters()), grp)
g1, i1, n1 = parallel.slider_groups(4)
assert g1 is None and (i1, n1) == (0, 1)
dist.destroy_process_group()
print("ok")
'''


def test_slider_groups_four_ranks_gloo(tmp_path):
    """More GPUs than one iteration can use: independent sliders side by side, each group a closed job."""
    script = tmp_path / "worker.py"
    script.write_text(_GROUPS_WORKER)
    port = 31500 + (os.getpid() % 2000)
    procs = [subprocess.Popen([sys.executable, str(script), ROOT, str(port), str(r)], stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(4)]
    outs = [p.communicate(timeout=240)[0] for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0 and "ok" in o, o


def test_launch_plan_dry_run_counts_and_flops():
    """Dry-run the SDXL forward on the meta device with shape-recording stand-ins for the kernels: the launch plan
    must contain every Linear/conv FLOP of SURVEY.md §8d (6.761 TFLOP per pass incl. attention) and the fusions
    DESIGN.md claims (one GEMM per fused QKV, cross-attention K/V batched, LoRA folded: no extra launches)."""
    import importlib
    import subprocess
    import sys as _sys

    code = (
        "import sys; sys.path.insert(0, %r); sys.path.insert(0, %r + '/tools');"
        "import shape_trace as st;"
        "tr = st.trace(2);"
        "import collections;"
        "k = collections.Counter(n for n, _, _ in tr);"
        "fl = sum(f for _, _, f in tr);"
        "print(len(tr), k['gemm_kernel'], k['attention_kernel'], k['layernorm_kernel'], fl)" % (ROOT, ROOT))
    out = subprocess.run([_sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    n, n_gemm, n_attn, n_ln, flops = out.stdout.strip().splitlines()[-1].split()
    assert int(n_attn) == 140 and int(n_ln) == 210
    # 743 Linear + 51 3x3/1x1 convs - fused QKV (2 x 70 saved) - batched cross K/V (140 -> 2) - small linears ...
    assert int(n_gemm) == 493
    assert int(n) == 1008
    per_pass = float(flops) / 2
    assert abs(per_pass - 6.761e12) / 6.761e12 < 0.01, per_pass


# ---------------------------------------------------------------------------------------- trainer host logic
def test_prompt_pair_loss_and_optimizer_factory():
    from sliders_b200 import trainer, train_util
    from sliders_b200.optim import AdamW

    g = torch.Generator().manual_seed(0)
    t, p, u, n = (torch.randn(1, 4, 8, 8, generator=g) for _ in range(4))
    mse = torch.nn.MSELoss()
    for action, sign in (("erase", -1.0), ("enhance", 1.0)):
        pair = trainer.PromptEmbedsPair(mse, None, None, None, None,
                                        trainer.PromptSettings(guidance_scale=4.0, action=action))
        got = pair.loss(target_latents=t, positive_latents=p, unconditional_latents=u, neutral_latents=n)
        assert torch.allclose(got, mse(t, n + sign * 4.0 * (p - u)))
    with pytest.raises(ValueError):
        trainer.PromptEmbedsPair(mse, None, None, None, None, trainer.PromptSettings(action="x")).loss(
            target_latents=t, positive_latents=p, unconditional_latents=u, neutral_latents=n)
    assert train_util.get_optimizer("AdamW") is AdamW and train_util.get_optimizer("adam") is torch.optim.Adam
    with pytest.raises(ValueError):
        train_util.get_optimizer("lion")
    for _ in range(20):
        h, w = train_util.get_random_resolution_in_bucket(1024)
        assert h % 64 == 0 and w % 64 == 0 and 512 <= h < 1024 and 512 <= w < 1024
    opt = torch.optim.SGD([torch.nn.Parameter(torch.zeros(1))], lr=1.0)
    for name in ("cosine", "cosine_with_restarts", "step", "constant", "linear"):
        assert train_util.get_lr_scheduler(name, opt, 1000, 1e-6) is not None
    with pytest.raises(ValueError):
        train_util.get_lr_scheduler("nope", opt, 1000, 1e-6)


def test_reference_prompt_pair_loss_matches_ours():
    """Against the reference's PromptEmbedsPair (prompt_util.py) on the same latents (golden, reference_calls.pt)."""
    from sliders_b200 import trainer

    fx = torch.load(os.path.join(GOLDEN, "reference_calls.pt"))["prompt_pair"]
    t, p, u, n = fx["target"], fx["positive"], fx["unconditional"], fx["neutral"]
    for action in ("erase", "enhance"):
        ref = fx[action]
        ours = trainer.PromptEmbedsPair(torch.nn.MSELoss(), None, None, None, None,
                                        trainer.PromptSettings(guidance_scale=fx["guidance_scale"], action=action,
                                                               batch_size=fx["batch_size"]))
        kw = dict(target_latents=t, positive_latents=p, unconditional_latents=u, neutral_latents=n)
        assert torch.equal(ref["loss"], ours.loss(**kw))
        assert (ref["batch_size"], ref["resolution"], ref["dynamic_crops"]) == (ours.batch_size, 512, ours.dynamic_crops)


_TRAIN_WORKER = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from sliders_b200 import trainer, train_util
world = int(sys.argv[4])
if world > 1:
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{sys.argv[2]}", rank=int(sys.argv[3]), world_size=world)

# stand-ins for the UNet call sites (the kernels need a GPU): any differentiable function of the adaptor weights
class Net(torch.nn.Module):
    def __init__(self):
        super().__init__()
        g = torch.Generator().manual_seed(5)
        self.a = torch.nn.Parameter(torch.randn(4, 4, generator=g) * 0.3)
        self.b = torch.nn.Parameter(torch.randn(4, generator=g) * 0.3)
        self.multiplier = 0.0
    def __enter__(self): self.multiplier = 1.0
    def __exit__(self, *a): self.multiplier = 0.0
net = Net()
calls = []
def predict_noise_xl(unet, sched, t, lat, text_embeddings, add_text_embeddings, add_time_ids, guidance_scale=7.5, **kw):
    calls.append("predict")
    e = text_embeddings.mean() + add_text_embeddings.mean()
    out = torch.tanh(lat.float() + e)
    if net.multiplier:
        out = out + net.multiplier * (torch.einsum("oc,bchw->bohw", net.a, lat.float()) + net.b[None, :, None, None])
    return out
def diffusion_xl(unet, sched, lat, text_embeddings, add_text_embeddings, add_time_ids, guidance_scale=1.0,
                 total_timesteps=1000, start_timesteps=0, cfg_split_group=False):
    calls.append("denoise")
    return lat * 0.9 + 0.01 * total_timesteps
train_util.predict_noise_xl, train_util.diffusion_xl = predict_noise_xl, diffusion_xl
from sliders_b200.scheduler import create_noise_scheduler
sched = create_noise_scheduler("ddim")
g = torch.Generator().manual_seed(1)
mk = lambda: trainer.PromptEmbedsXL(torch.randn(1, 77, 8, generator=g), torch.randn(1, 4, generator=g))
unc, tgt, pos, neu = mk(), mk(), mk(), mk()
pair = trainer.PromptEmbedsPair(torch.nn.MSELoss(), tgt, pos, unc, neu,
                                trainer.PromptSettings(guidance_scale=2.0, resolution=64, batch_size=2, action="erase"))
opt = torch.optim.AdamW(net.parameters(), lr=1e-2)
losses = []
for it in range(3):
    gen = torch.Generator().manual_seed(100 + it + (dist.get_rank() if world > 1 else 0))  # ranks draw DIFFERENT noise
    losses.append(float(trainer.text_slider_step_xl(None, net, sched, opt, None, pair, timesteps_to=None if it else 7,
                                                    device="cpu", weight_dtype=torch.float32, generator=gen)))
torch.save({"a": net.a.detach(), "b": net.b.detach(), "losses": losses, "calls": calls}, sys.argv[5])
if world > 1:
    dist.destroy_process_group()
print("ok")
'''


def test_text_slider_step_sharded_two_ranks_gloo(tmp_path):
    """BASELINE config 3's host logic on CPU: with the four predictions sharded over 2 ranks the replicas end with
    identical adaptor weights, each rank runs only its share of the predictions, and rank 0's trajectory equals the
    single-process one (rank 0's noise is broadcast)."""
    script = tmp_path / "train_worker.py"
    script.write_text(_TRAIN_WORKER)
    port = 31500 + (os.getpid() % 2000)
    outs = [str(tmp_path / f"out{r}.pt") for r in range(2)]
    procs = [subprocess.Popen([sys.executable, str(script), ROOT, str(port), str(r), "2", outs[r]],
                              stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True) for r in range(2)]
    logs = [p.communicate(timeout=300)[0] for p in procs]
    for p, o in zip(procs, logs):
        assert p.returncode == 0 and "ok" in o, o
    single = str(tmp_path / "single.pt")
    p = subprocess.run([sys.executable, str(script), ROOT, str(port + 1), "0", "1", single], capture_output=True,
                       text=True, timeout=300)
    assert p.returncode == 0, p.stdout + p.stderr
    r0, r1, s = torch.load(outs[0]), torch.load(outs[1]), torch.load(single)
    assert torch.equal(r0["a"], r1["a"]) and torch.equal(r0["b"], r1["b"])
    assert r0["losses"] == r1["losses"]
    # iteration 0 has a fixed step count and rank 0's noise: same loss as the single process
    assert abs(r0["losses"][0] - s["losses"][0]) < 1e-6
    # rank 1 owns the grad-carrying target prediction (forward + backward), rank 0 the three frozen ones
    assert r0["calls"].count("predict") == 9 and r1["calls"].count("predict") == 3
    assert s["calls"].count("predict") == 12


_IMG_WORKER = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from sliders_b200 import trainer, train_util
world = int(sys.argv[4])
if world > 1:
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{sys.argv[2]}", rank=int(sys.argv[3]), world_size=world)

class Net(torch.nn.Module):
    def __init__(self):
        super().__init__()
        g = torch.Generator().manual_seed(5)
        self.a = torch.nn.Parameter(torch.randn(4, 4, generator=g) * 0.3)
        self.multiplier, self.lora_scale = 0.0, 1.0
    def set_lora_slider(self, scale): self.lora_scale = scale
    def __enter__(self): self.multiplier = self.lora_scale
    def __exit__(self, *a): self.multiplier = 0.0
net = Net()
def predict_noise_xl(unet, sched, t, lat, text_embeddings, add_text_embeddings, add_time_ids, guidance_scale=7.5, **kw):
    assert text_embeddings.shape[0] == 2 * lat.shape[0] and add_time_ids.shape[0] == 2 * lat.shape[0]
    e = text_embeddings[lat.shape[0]:].mean(dim=(1, 2))[:, None, None, None]
    return torch.tanh(lat.float() + e) + net.multiplier * torch.einsum("oc,bchw->bohw", net.a, lat.float())
train_util.predict_noise_xl = predict_noise_xl
from sliders_b200.scheduler import create_noise_scheduler
sched = create_noise_scheduler("ddim")
g = torch.Generator().manual_seed(1)
mk = lambda: trainer.PromptEmbedsXL(torch.randn(1, 77, 8, generator=g), torch.randn(1, 4, generator=g))
unc, pos, neu = mk(), mk(), mk()
bs = int(sys.argv[6])
pair = trainer.PromptEmbedsPair(torch.nn.MSELoss(), pos, pos, unc, neu,
                                trainer.PromptSettings(guidance_scale=1.0, resolution=64, batch_size=bs))
low = torch.randn(bs, 4, 8, 8, generator=g); high = low + 0.2 * torch.randn(bs, 4, 8, 8, generator=g)
opt = torch.optim.SGD(net.parameters(), lr=0.1)
out = []
for it in range(2):
    ls = trainer.image_slider_step_xl(None, net, sched, opt, None, pair, low, high, 2.0, timesteps_to=10, seed=3 + it,
                                      device="cpu", weight_dtype=torch.float32)
    out.append([float(l) for l in ls])
torch.save({"a": net.a.detach(), "losses": out}, sys.argv[5])
if world > 1:
    dist.destroy_process_group()
print("ok")
'''


@pytest.mark.parametrize("world,bs", [(2, 1), (4, 2)])
def test_image_slider_step_sharded_gloo(tmp_path, world, bs):
    """BASELINE config 4's host logic: the +scale / -scale predictions on rank parity (and the batch split over
    rank // 2 when it divides) give the single-process weights."""
    script = tmp_path / "img_worker.py"
    script.write_text(_IMG_WORKER)
    port = 33500 + (os.getpid() % 2000) + 7 * world
    outs = [str(tmp_path / f"o{r}.pt") for r in range(world)]
    procs = [subprocess.Popen([sys.executable, str(script), ROOT, str(port), str(r), str(world), outs[r], str(bs)],
                              stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True) for r in range(world)]
    logs = [p.communicate(timeout=300)[0] for p in procs]
    for p, o in zip(procs, logs):
        assert p.returncode == 0 and "ok" in o, o
    single = str(tmp_path / "single.pt")
    p = subprocess.run([sys.executable, str(script), ROOT, str(port + 1), "0", "1", single, str(bs)],
                       capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stdout + p.stderr
    ref = torch.load(single)
    for o in outs:
        got = torch.load(o)
        assert torch.allclose(got["a"], ref["a"], rtol=1e-5, atol=1e-6), (got["a"] - ref["a"]).abs().max()
        assert all(abs(x - y) < 1e-5 for a, b in zip(got["losses"], ref["losses"]) for x, y in zip(a, b))


def test_euler_scheduler_matches_oracle_restatement():
    """sliders_b200.scheduler.EulerDiscreteScheduler (eval loop, generate_images_xl.py:267-358) against oracle/euler.py."""
    from oracle import euler as oeuler
    from sliders_b200 import scheduler as psched

    for spacing, offset in (("leading", 1), ("linspace", 0), ("trailing", 0)):
        a = psched.EulerDiscreteScheduler(timestep_spacing=spacing, steps_offset=offset)
        b = oeuler.EulerDiscreteScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear",
                                          timestep_spacing=spacing, steps_offset=offset)
        assert abs(float(a.init_noise_sigma) - float(b.init_noise_sigma)) < 1e-4
        for n in (50, 30, 7):
            a.set_timesteps(n)
            b.set_timesteps(n)
            assert torch.equal(a.timesteps, b.timesteps) and torch.allclose(a.sigmas, b.sigmas)
            g = torch.Generator().manual_seed(n)
            x = torch.randn(2, 4, 8, 8, generator=g) * float(a.init_noise_sigma)
            for t in a.timesteps_host[:4] + a.timesteps_host[-2:]:
                e = torch.randn(2, 4, 8, 8, generator=g)
                assert torch.allclose(a.scale_model_input(x, t), b.scale_model_input(x, t), atol=1e-6)
                assert torch.allclose(a.step(e, t, x).prev_sample, b.step(e, t, x).prev_sample, atol=1e-5)
    assert isinstance(psched.create_noise_scheduler("euler"), psched.EulerDiscreteScheduler)


def test_lms_scheduler_matches_oracle_restatement():
    """sliders_b200.scheduler.LMSDiscreteScheduler (eval-scripts/generate_images_sd1.py:51,169-192) against oracle/lms.py
    over a whole 12-step trajectory (the multistep history makes every step depend on the previous ones)."""
    from oracle import lms as olms
    from sliders_b200 import scheduler as psched

    a = psched.create_noise_scheduler("lms")
    b = olms.LMSDiscreteScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear")
    assert isinstance(a, psched.LMSDiscreteScheduler) and a.step_kind == "generic"
    a.set_timesteps(12)
    b.set_timesteps(12)
    assert torch.equal(a.timesteps, b.timesteps) and torch.allclose(a.sigmas, b.sigmas)
    assert abs(float(a.init_noise_sigma) - float(b.init_noise_sigma)) < 1e-4
    g = torch.Generator().manual_seed(2)
    xa = xb = torch.randn(2, 4, 8, 8, generator=g) * float(a.init_noise_sigma)
    for t in a.timesteps_host:
        e = torch.randn(2, 4, 8, 8, generator=g)
        assert torch.allclose(a.scale_model_input(xa, t), b.scale_model_input(xb, t), atol=1e-5)
        xa = a.step(e, t, xa).prev_sample
        xb = b.step(e, t, xb).prev_sample
        assert torch.allclose(xa, xb, rtol=1e-4, atol=1e-4)


def test_io_unet_and_slider_ingestion(tmp_path):
    """sliders_b200.io: an HF-style UNet state dict (safetensors) and slider checkpoints written by the reference-style
    `save_weights` load back bit for bit; mismatching files fail loudly."""
    from safetensors.torch import save_file

    from oracle import unet as ounet
    from sliders_b200 import io as sio, lora as plora, synthetic
    from sliders_b200.unet import UNet2DConditionModel, UNetConfig

    cfg = UNetConfig.from_dict(ounet.UNetConfig.tiny_xl().__dict__)
    src = UNet2DConditionModel(cfg)
    synthetic.init_synthetic_(src, seed=3)
    f = str(tmp_path / "diffusion_pytorch_model.safetensors")
    save_file({k: v.contiguous() for k, v in src.state_dict().items()}, f)
    got = sio.load_unet(cfg, f, dtype=torch.float32)
    for (k, a), (_, b) in zip(src.state_dict().items(), got.state_dict().items()):
        assert torch.equal(a, b), k
    with pytest.raises(RuntimeError, match="not a UNet2DConditionModel state dict"):
        sio.load_unet(UNetConfig.from_dict(ounet.UNetConfig.tiny_sd().__dict__), f)
    net = plora.LoRANetwork(src, rank=4, multiplier=1.0, alpha=1.0, train_method="noxattn")
    synthetic.init_lora_nonzero_(net, seed=4, up_std=0.05)
    for ext in (".pt", ".safetensors"):
        ck = str(tmp_path / ("slider" + ext))
        net.save_weights(ck, dtype=torch.bfloat16)
        other = UNet2DConditionModel(cfg)
        net2 = plora.LoRANetwork(other, rank=4, multiplier=1.0, alpha=1.0, train_method="noxattn")
        sio.load_slider(net2, ck)
        for (k, a), (_, b) in zip(net.state_dict().items(), net2.state_dict().items()):
            assert torch.equal(a.to(torch.bfloat16).float(), b.float()), k
        net8 = plora.LoRANetwork(UNet2DConditionModel(cfg), rank=8, multiplier=1.0, alpha=1.0, train_method="noxattn")
        with pytest.raises(RuntimeError, match="shape"):
            sio.load_slider(net8, ck)
        netx = plora.LoRANetwork(UNet2DConditionModel(cfg), rank=4, multiplier=1.0, alpha=1.0, train_method="xattn")
        with pytest.raises(RuntimeError, match="adaptor keys"):
            sio.load_slider(netx, ck)


def test_slice_tape_and_rank_assignment():
    """Host pieces of the backward / sharding logic that need no GPU: batch slicing of a tape (autograd.slice_tape) and
    the condition -> rank assignment of the sharded text-slider step."""
    from sliders_b200.autograd import slice_tape

    B = 2
    rec = ("res", (object(), torch.arange(2 * 3 * 3 * 8).view(2, 3, 3, 8), None, torch.zeros(2, 16), torch.ones(2, 32, 2),
                   torch.arange(2 * 9 * 4).view(18, 4), [torch.zeros(2 * 77, 6), 77, None]))
    tape = [("scales", {1: ("a", 0.25)}), rec, ("skip", None)]
    out = slice_tape(tape, 1, 2, B)
    assert out[0] == tape[0] and out[2] == ("skip", None)
    r = out[1][1]
    assert r[0] is rec[1][0] and r[2] is None
    assert r[1].shape == (1, 3, 3, 8) and torch.equal(r[1], rec[1][1][1:2])
    assert r[3].shape == (1, 16) and r[4].shape == (1, 32, 2)
    assert torch.equal(r[5], rec[1][5][9:18])            # token matrix [B * 9, C]: rows of sample 1
    assert r[6][0].shape == (77, 6) and r[6][1] == 77
    with pytest.raises(RuntimeError):
        slice_tape(torch.zeros(5), 1, 2, B)               # not batch-major
    # views, not copies
    assert r[1].data_ptr() == rec[1][1][1:2].data_ptr()

    # owner mapping of text_slider_step_xl: the grad-carrying prediction gets the last rank, the frozen ones the others
    def owners(world):
        o = {"target": world - 1}
        for i, name in enumerate(("positive", "neutral", "unconditional")):
            o[name] = i % max(world - 1, 1)
        return o

    assert owners(1) == {"target": 0, "positive": 0, "neutral": 0, "unconditional": 0}
    assert owners(2) == {"target": 1, "positive": 0, "neutral": 0, "unconditional": 0}
    assert owners(4) == {"target": 3, "positive": 0, "neutral": 1, "unconditional": 2}
    assert owners(8)["target"] == 7 and set(owners(8).values()) == {0, 1, 2, 7}
    import inspect

    from sliders_b200 import trainer
    src = inspect.getsource(trainer.text_slider_step_xl)
    assert 'owner = {"target": world - 1}' in src and "i % max(world - 1, 1)" in src  # the mapping tested above is the shipped one


def test_image_slider_step_sd_host_logic(monkeypatch):
    """`trainer.image_slider_step` (train_lora-scale.py:185-330) with a differentiable stand-in for the UNet call site:
    both signs are applied, gradients of the two losses accumulate, the optimizer steps once."""
    from sliders_b200 import trainer, train_util
    from sliders_b200.scheduler import create_noise_scheduler

    class Net(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.a = torch.nn.Parameter(torch.full((4, 4), 0.1))
            self.multiplier, self.lora_scale, self.seen = 0.0, 1.0, []

        def set_lora_slider(self, scale):
            self.lora_scale = scale

        def __enter__(self):
            self.multiplier = self.lora_scale
            self.seen.append(self.lora_scale)

        def __exit__(self, *a):
            self.multiplier = 0.0

    net = Net()
    calls = []

    def predict_noise(unet, sched, t, lat, emb, guidance_scale=7.5):
        assert emb.shape[0] == 2 * lat.shape[0] and guidance_scale == 1
        calls.append(float(emb[lat.shape[0]:].mean()))
        return torch.tanh(lat.float()) + net.multiplier * torch.einsum("oc,bchw->bohw", net.a, lat.float())

    monkeypatch.setattr(train_util, "predict_noise", predict_noise)
    g = torch.Generator().manual_seed(0)
    unc, pos, neu = (torch.randn(1, 77, 8, generator=g) for _ in range(3))
    pair = trainer.PromptEmbedsPair(torch.nn.MSELoss(), pos, pos, unc, neu, trainer.PromptSettings(batch_size=2))
    low = torch.randn(2, 4, 8, 8, generator=g)
    high = low + 0.1
    opt = torch.optim.SGD(net.parameters(), lr=0.5)
    before = net.a.detach().clone()
    losses = trainer.image_slider_step(None, net, create_noise_scheduler("ddim"), opt, None, pair, low, high, 3.0,
                                       timesteps_to=10, seed=1, device="cpu", weight_dtype=torch.float32)
    assert net.seen == [3.0, -3.0] and len(calls) == 2 and len(losses) == 2
    assert abs(calls[0] - float(pos.mean())) < 1e-6 and abs(calls[1] - float(neu.mean())) < 1e-6
    assert not torch.equal(before, net.a.detach()) and net.multiplier == 0.0
    calls.clear()
    trainer.image_slider_step(None, net, create_noise_scheduler("ddim"), opt, None, pair, low, high, 3.0, timesteps_to=10,
                              seed=1, device="cpu", weight_dtype=torch.float32, reference_dead_code=True)
    assert len(calls) == 4


def test_stochastic_schedulers_match_oracle_restatement():
    """`train.noise_scheduler: "ddpm" | "euler_a"` (model_util.py:247-278): sliders_b200.scheduler against
    oracle/stochastic.py over whole trajectories with the same generator stream."""
    from oracle import stochastic as ost
    from sliders_b200 import scheduler as psched

    kw = dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear")
    pairs = ((psched.create_noise_scheduler("ddpm"), ost.DDPMScheduler(clip_sample=False, **kw)),
             (psched.create_noise_scheduler("euler_a"), ost.EulerAncestralDiscreteScheduler(**kw)))
    assert isinstance(pairs[0][0], psched.DDPMScheduler) and isinstance(pairs[1][0], psched.EulerAncestralDiscreteScheduler)
    for a, b in pairs:
        assert a.step_kind == "affine+noise"
        assert abs(float(a.init_noise_sigma) - float(b.init_noise_sigma)) < 1e-4
        for n in (50, 11):
            a.set_timesteps(n)
            b.set_timesteps(n)
            assert torch.equal(a.timesteps.double(), b.timesteps.double())
            g = torch.Generator().manual_seed(n)
            x0 = torch.randn(2, 4, 8, 8, generator=g) * float(a.init_noise_sigma)
            xa = xb = x0
            ga, gb = torch.Generator().manual_seed(5), torch.Generator().manual_seed(5)
            for t in a.timesteps_host:
                e = torch.randn(2, 4, 8, 8, generator=g)
                assert torch.allclose(a.scale_model_input(xa, t), b.scale_model_input(xb, t), atol=1e-5)
                xa = a.step(e, t, xa, generator=ga).prev_sample
                xb = b.step(e, t, xb, generator=gb).prev_sample
                assert torch.allclose(xa, xb, rtol=1e-4, atol=1e-4), (type(a).__name__, n, t)
    # the noise term is really there (and absent at the last DDPM step, t = 0)
    d = pairs[0][0]
    d.set_timesteps(1000)
    assert d._noise_std(0) == 0.0 and d._noise_std(500) > 0.0
    with pytest.raises(ValueError):
        psched.create_noise_scheduler("plms")


def test_second_network_on_one_unet_is_refused():
    """ADVICE r1: the reference chains `org_forward`, so two LoRANetworks on one UNet both apply; the fused kernels carry
    one adaptor per leaf, so the engine must refuse instead of silently dropping the first network."""
    from sliders_b200 import lora as plora
    from sliders_b200.unet import UNet2DConditionModel, UNetConfig

    from oracle import unet as ounet

    pm = UNet2DConditionModel(UNetConfig.from_dict(ounet.UNetConfig.tiny_xl().__dict__))
    plora.LoRANetwork(pm, rank=4, alpha=1.0, train_method="noxattn")
    assert len(pm._adapted_leaves()) > 0
    plora.LoRANetwork(pm, rank=4, alpha=1.0, train_method="noxattn")
    pm.__dict__.pop("_adapted_cache", None)
    with pytest.raises(RuntimeError, match="second LoRANetwork"):
        pm._adapted_leaves()
