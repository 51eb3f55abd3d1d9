"""Row (b) of SURVEY.md §8 — the drop-in boundary — checked against the REFERENCE'S OWN trainer code.  The fused model runs on CPU
with emulated kernels (tests/emu_lib.py): what is under test is the interface, not the arithmetic.

Where the reference computes something (rotary tables, sampling schedule, loss / parameter trajectories, gradients, an embedding cache,
validation-loop latents), its results are stored in tests/golden/boundary_golden.pt (generator: tests/golden/make_boundary_golden.py)
and the fused path is compared with them; the trainer the fused step is patched into is then a plain object carrying what
`patch_trainer` reads, and the oracle (pinned to the reference by tests/test_reference_goldens.py) stands in for the reference module.
Where the reference's trainer plumbing (`BaseTrainer.add_lora_adapter`, `.load_pretrain_lora_model`, `.save_lora`,
`.setup_model_device_train_mode`, `.configure_optimizers`, `.accelerator_prepare`, `.train_epoch`) acts on the transformer, the tests
make the calls it makes (cited by line), with `diffusers` / `peft` / `accelerate` from tests/shims; the files it writes and the facts
about its trainer classes are part of the stored golden."""
import os
import sys
import types

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))

sys.path.insert(0, os.path.join(HERE, "golden"))
sys.path.insert(0, os.path.join(HERE, "shims"))


@pytest.fixture(scope="module")
def golden():
    return torch.load(os.path.join(HERE, "golden", "boundary_golden.pt"))


@pytest.fixture(scope="module")
def shims():
    """`diffusers` / `peft` / `accelerate` from tests/shims (restatements of their published behaviour)."""
    import stub_importer
    return stub_importer.install()


@pytest.fixture()
def emu():
    import emu_lib
    from qflux_b200 import lib
    restore = emu_lib.install(lib)
    yield
    restore()


def _cfg(r=4, alpha=8, targets=("to_q", "to_k", "to_v", "to_out.0"), pretrained=None):
    lora = types.SimpleNamespace(r=r, lora_alpha=alpha, init_lora_weights="gaussian", target_modules=list(targets), pretrained_weight=pretrained)
    return types.SimpleNamespace(model=types.SimpleNamespace(lora=lora), train=types.SimpleNamespace(max_grad_norm=0.5, gradient_accumulation_steps=1))


def _fused(host_only=True):
    import ref_common as rc
    from qflux_b200.qwen_model import QwenB200Config, QwenImageB200
    c = rc.QWEN_HD128
    return QwenImageB200(QwenB200Config(num_layers=c["num_layers"], num_attention_heads=c["num_attention_heads"],
                                        joint_attention_dim=c["joint_attention_dim"]), device="cpu", _host_only=host_only)


def _reference_module(case):
    """The oracle with the reference's weights (filled by name) and a PEFT-style `peft_config`: what `from_reference` / `patch_trainer`
    read off a loaded reference transformer."""
    import ref_common as rc
    sys.path.insert(0, HERE)
    from test_reference_goldens import _oracle
    spec = rc.CASES[case]
    orc, _ = _oracle(spec)
    orc.peft_config = {"default": types.SimpleNamespace(r=spec["r"], lora_alpha=spec["alpha"], target_modules=spec["targets"],
                                                        init_lora_weights="gaussian")}
    return orc


def _patched_trainer(case, criterion_name):
    """A trainer object as `patch_trainer` sees it (dit, criterion, config.train, accelerator), patched."""
    from qflux_b200 import patch_trainer
    tr = types.SimpleNamespace(dit=_reference_module(case), criterion=type(criterion_name, (), {})(), config=_cfg(),
                               accelerator=types.SimpleNamespace(device=torch.device("cpu")), vae_scale_factor=8)
    return patch_trainer(tr, _host_only=True)


def _lora_rel(got, want):
    assert set(want) <= set(got)
    num = sum(((got[n].float() - want[n].float()) ** 2).sum() for n in want)
    return float((num / sum((v.float() ** 2).sum() for v in want.values())).sqrt())


def _lora_modules(model):
    """Every sub-module whose qualified name contains "lora": what the reference's `get_lora_layers` (lora_utils.py:25-38) collects
    for `accelerator_prepare` to wrap (AttnProcsLayers) or to list as FSDP `ignored_modules` (base_trainer.py:340-342, 383-387)."""
    return {n: mod for n, mod in model.named_modules() if "lora" in n}


def test_reference_add_lora_adapter_and_module_scan(shims, emu):
    """What base_trainer.py:929-941 does to the transformer — `add_adapter(LoraConfig(r, lora_alpha, init_lora_weights, target_modules),
    adapter_name=...)` then `set_adapter(adapter_name)` — on the fused model; the LoRA module scan finds child modules whose parameters
    are exactly the trainable LoRA parameters."""
    from peft import LoraConfig
    m = _fused()
    lora = _cfg().model.lora
    m.add_adapter(LoraConfig(r=lora.r, lora_alpha=lora.lora_alpha, init_lora_weights=lora.init_lora_weights,
                             target_modules=lora.target_modules), adapter_name="lora_edit")
    m.set_adapter("lora_edit")
    names = [n for n, _ in m.named_parameters()]
    assert len(names) == 2 * 4 * 2 and all(".lora_A.lora_edit.weight" in n or ".lora_B.lora_edit.weight" in n for n in names)
    assert all(p.requires_grad for p in m.parameters()) and all("lora" in n for n in names)  # qwen_image_edit_trainer.py:314-318
    assert set(m.peft_config) == {"lora_edit"} and m.peft_config["lora_edit"].r == 4
    layers = _lora_modules(m)
    assert layers and all(isinstance(v, torch.nn.Module) for v in layers.values())
    found = {id(p) for v in layers.values() for p in v.parameters()}
    assert found == {id(p) for p in m.parameters()}
    with pytest.raises(Exception):
        m.set_adapter("other")
    m.set_adapter("lora_edit")
    assert m.to("cpu") is m and m.to(torch.bfloat16) is m  # no-op moves are accepted (base_trainer.py:388) ...
    with pytest.raises(Exception):
        m.to(torch.float32)                                  # ... re-typing the fused HBM layout is refused loudly


def test_pos_embed_matches_reference_rope(golden):
    """`dit.pos_embed([shapes], [T], device)` (qwen_image_edit_trainer.py:734) vs the reference's QwenEmbedRope (scale_rope=True)."""
    m = _fused()
    cases = (([(1, 4, 4), (1, 4, 4)], 7), ([(1, 4, 6), (1, 4, 6), (1, 2, 8)], 11))
    for (shapes, T), (b_v, b_t) in zip(cases, golden["rope"], strict=True):
        a_v, a_t = m.pos_embed([shapes], [T], device=torch.device("cpu"))
        assert a_v.shape == b_v.shape and a_t.shape == b_t.shape
        assert (a_v - b_v).abs().max() < 2e-5 and (a_t - b_t).abs().max() < 2e-5


def test_patch_trainer_runs_the_reference_loop_body(golden, emu):
    """patch_trainer on a trainer object: the reference's loop body (training_step -> backward -> clip_gradients (global-norm clip at
    train.max_grad_norm) -> optimizer.step -> zero_grad, base_trainer.py:518-533) on the fused model tracks the stored un-patched
    reference run (its losses and LoRA parameters after three AdamW steps)."""
    import ref_common as rc
    from qflux_b200.mmdit_base import FusedMMDiTBase
    x = rc.rand_inputs(rc.CASES["qwen_hd128"])
    emb = {k: v for k, v in x.items() if k != "u"}
    tr = _patched_trainer("qwen_hd128", "MseLoss")
    assert isinstance(tr.dit, FusedMMDiTBase) and tr.dit.peft_config["default"].r == 4
    params = [p for p in tr.dit.parameters() if p.requires_grad]
    tr.optimizer = torch.optim.AdamW(params, lr=1e-2, weight_decay=0.0)
    l_b = []
    for it in range(3):
        torch.manual_seed(100 + it)
        e = dict(emb)  # the reference draws randn_like(image_latents) in fp32 on the CPU: hand the fused step the same draw
        e["noise"] = torch.randn_like(emb["image_latents"])
        e["u"] = x["u"]
        loss = tr._compute_loss(e)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(params, tr.config.train.max_grad_norm)
        tr.optimizer.step()
        tr.optimizer.zero_grad()
        l_b.append(float(loss))
    l_r, p_r = golden["loop_body"]["losses"], golden["loop_body"]["params"]
    p_b = {n: p.detach().float().clone() for n, p in tr.dit.named_parameters() if p.requires_grad}
    assert all(abs(a - b) < 2e-2 for a, b in zip(l_r, l_b, strict=True)), (l_r, l_b)
    assert l_b[-1] < l_b[0]  # the optimizer actually moved the LoRA parameters in the right direction
    assert set(p_r) == set(p_b)
    assert _lora_rel(p_b, p_r) < 2e-2  # bf16 parameters vs the fp32 reference run after three AdamW steps


def _safetensors_header(path):
    import json
    import struct
    with open(path, "rb") as f:
        return json.loads(f.read(struct.unpack("<Q", f.read(8))[0]))


def test_save_lora_roundtrip_through_reference_code(golden, shims, emu, tmp_path):
    """save_lora (base_trainer.py:858-875: get_peft_model_state_dict -> convert_state_dict_to_diffusers -> pipeline.save_lora_weights ->
    safetensors) on the fused model writes the file the reference's own save_lora wrote (stored header: keys, dtypes, shapes, layout;
    the reference classified it "PEFT"); the file loads back into the fused model, its keys are the LoRA parameter names the reference
    model had after its `load_lora_adapter` (:983), and the resume path of `load_pretrain_lora_model` (:943-1002: add_lora_adapter ->
    load_state_dict(strict=False) -> no unexpected keys) restores the factors."""
    import ref_common as rc
    import safetensors.torch
    from diffusers import FluxKontextPipeline
    from diffusers.utils import convert_state_dict_to_diffusers
    from peft import LoraConfig
    from peft.utils import get_peft_model_state_dict
    want_file = golden["save_lora"]

    def with_adapter(name="default"):
        m = _fused()
        lora = _cfg().model.lora
        m.add_adapter(LoraConfig(r=lora.r, lora_alpha=lora.lora_alpha, init_lora_weights=lora.init_lora_weights,
                                 target_modules=lora.target_modules), adapter_name=name)
        m.set_adapter(name)
        return m
    m = with_adapter()
    rc.det_fill_(type("B", (), {"named_parameters": lambda s: iter(m._lora_params.items())})(), 5)
    folder = str(tmp_path / "ckpt")
    FluxKontextPipeline.save_lora_weights(folder, convert_state_dict_to_diffusers(get_peft_model_state_dict(m, adapter_name="default")),
                                          safe_serialization=True)
    path = os.path.join(folder, "pytorch_lora_weights.safetensors")
    assert _safetensors_header(path) == want_file["header"] and want_file["kind"] == "PEFT"
    sd = safetensors.torch.load_file(path)
    assert len(sd) == 16 and all(k.startswith("transformer.") and (k.endswith(".lora_A.weight") or k.endswith(".lora_B.weight")) for k in sd)
    want = {n: p.detach().clone() for n, p in m.named_parameters()}
    assert all(torch.equal(sd["transformer." + n.replace(".default.", ".")], v) for n, v in want.items())
    # (1) into a fresh fused model through the diffusers entry point
    m2 = _fused()
    m2.load_lora_adapter(path, adapter_name="default")
    assert m2.lora_rank == 4 and all(torch.equal(p, want[n]) for n, p in m2.named_parameters())
    # (2) the reference model held exactly these parameter names after loading the file
    assert want_file["reference_lora_names"] == sorted(want)
    # (3) the trainer's resume path
    m3 = with_adapter()
    missing, unexpected = m3.load_state_dict(safetensors.torch.load_file(path), strict=False)
    assert not unexpected
    assert all(torch.equal(p, want[n]) for n, p in m3.named_parameters())
    # state_dict() hands out compact tensors (safetensors refuses views), torch.save stays small
    assert all(v.is_contiguous() for v in m.state_dict().values() if v.ndim == 2 and v.shape[1] == 4)


def test_fused_adamw_honours_the_optimizer_contract(emu):
    """ADVICE r1: `step(closure=None)` positional contract, AcceleratedOptimizer-style wrappers (`.optimizer`), mean over ranks x micro-steps."""
    import ref_common as rc
    from qflux_b200.optim import FusedLoraAdamW
    from qflux_b200.train_step import QwenImageEditStep, _sync_and_step
    sys.path.insert(0, HERE)
    from test_reference_goldens import _b200_model
    m, _ = _b200_model(rc.CASES["qwen_hd128"], "cpu", True)  # name-derived non-zero weights (an all-zero model has zero LoRA gradients)
    opt = FusedLoraAdamW(m, lr=1e-2)

    class Wrapped:  # accelerate.optimizer.AcceleratedOptimizer: forwards step(closure) to .optimizer
        def __init__(self, o):
            self.optimizer = o

        def step(self, closure=None):
            return self.optimizer.step(closure)
    x = rc.rand_inputs(rc.CASES["qwen_hd128"])
    emb = {k: x[k] for k in ("image_latents", "control_latents", "prompt_embeds", "img_shapes")}
    step = QwenImageEditStep(m, "mse", max_grad_norm=1.0)
    before = [p.detach().clone() for p in m.parameters()]
    step.train_step(emb, Wrapped(opt), noise=torch.randn(2, 16, 64).bfloat16(), u=x["u"])
    assert opt.step_count == 1 and any(not torch.equal(a, b) for a, b in zip(before, m.parameters()))
    assert opt.step(None) is None and opt.step_count == 2          # positional closure slot accepts None
    assert opt.step(lambda: torch.tensor(3.0)).item() == 3.0        # and a real closure
    # the divisor set by the sync (world x micro-steps) is what a later plain step() uses: a summed gradient is never applied as-is
    m.G32.fill_(2.0)
    _sync_and_step(m, opt, 0.0, micro_steps=4)
    assert opt.grad_divisor == 4 and abs(float(opt.grad_norm_sq.sqrt()) - 0.5 * m.G32.numel() ** 0.5) < 1e-2 * m.G32.numel() ** 0.5


def test_patch_trainer_flux_shared_and_multires(golden, emu):
    """patch_trainer on the FLUX-Kontext trainer: the reference's `embeddings` dict (pixel `image`, pixel-space `img_shapes`, `control_ids`)
    goes through the fused step unchanged, in shared mode (flux_kontext_trainer.py:494-577) and in multi-resolution mode (:579-796), and
    gives the stored loss and LoRA gradients of the reference trainer's `_compute_loss`."""
    import ref_common as rc
    for case, crit in (("flux_hd128", "MseLoss"), ("flux_custom_multires", "AttentionMaskMseLoss")):
        spec, want = rc.CASES[case], golden["flux_train"][case]
        x = rc.rand_inputs(spec)
        e = {k: v for k, v in x.items() if k not in ("img_shapes_latent", "hw")}
        if spec["kind"] == "flux":
            h_, w_ = x["hw"]
            e["control_ids"] = want["control_ids"]  # the reference's _prepare_latent_image_ids with 1 in the first column
            e["img_shapes"] = [[(3, h_ * 16, w_ * 16), (3, h_ * 16, w_ * 16)]] * spec["B"]
        else:  # the fused step takes one padded noise tensor and a flat timestep vector
            lt = [s[0][1] * s[0][2] for s in x["img_shapes_latent"]]
            nz = torch.zeros(len(lt), max(lt), 64)
            for b, n in enumerate(lt):
                nz[b, :n] = x["noise"][b]
            e["noise"], e["timestep"] = nz, x["timestep"]
        tr = _patched_trainer(case, crit)
        loss = tr._compute_loss(e)
        loss.backward()
        g_b = {n: p.grad.float().clone() for n, p in tr.dit.named_parameters() if p.requires_grad and p.grad is not None}
        assert abs(want["loss"] - float(loss)) < 1e-2, (case, want["loss"], float(loss))
        assert _lora_rel(g_b, want["grads"]) < 2e-2, case


def test_sampler_schedule_matches_reference_prepare_predict_timesteps(golden):
    """§8 f2: `flow_match_sigmas` vs the stored results of the reference's `BaseTrainer.prepare_predict_timesteps` (base_trainer.py:1009-1043
    -> calculate_shift, retrieve_timesteps -> FlowMatchEulerDiscreteScheduler.set_timesteps(sigmas=, mu=)), for the Qwen-Image and the
    FLUX scheduler configs, and the Euler update vs its `scheduler.step`."""
    from qflux_b200.sampler import _euler_step, calculate_shift, flow_match_sigmas
    qwen = dict(num_train_timesteps=1000, shift=1.0, use_dynamic_shifting=True, base_shift=0.5, max_shift=0.9, base_image_seq_len=256,
                max_image_seq_len=8192, shift_terminal=0.02)
    flux = dict(num_train_timesteps=1000, shift=3.0, use_dynamic_shifting=True, base_shift=0.5, max_shift=1.15, base_image_seq_len=256,
                max_image_seq_len=4096)
    cases = [(conf, steps, seq) for conf in (qwen, flux) for steps, seq in ((20, 1024), (8, 4096), (50, 400))]
    g = torch.Generator().manual_seed(9)  # the draws the stored Euler steps were taken on
    for (conf, steps, seq), r in zip(cases, golden["schedule"], strict=True):
        x, v = torch.randn(2, 8, 64, generator=g).bfloat16(), torch.randn(2, 8, 64, generator=g).bfloat16()
        assert (r["steps"], r["seq"]) == (steps, seq)
        assert abs(calculate_shift(seq, conf["base_image_seq_len"], conf["max_image_seq_len"], conf["base_shift"], conf["max_shift"])
                   - r["shift"]) < 1e-12
        sig = flow_match_sigmas(steps, seq, base_seq_len=conf["base_image_seq_len"], max_seq_len=conf["max_image_seq_len"],
                                base_shift=conf["base_shift"], max_shift=conf["max_shift"], shift_terminal=conf.get("shift_terminal"))
        assert r["n"] == steps and sig.numel() == steps + 1 and sig[-1] == 0
        assert torch.allclose(sig[:-1] * 1000, r["timesteps"], rtol=2e-6, atol=1e-4), (conf, steps, seq)
        assert torch.allclose(sig, r["sigmas"], rtol=2e-6, atol=1e-7)
        # one Euler step of the loop in sampler.py == scheduler.step (fp32 update, model dtype out)
        assert torch.equal(r["euler_step"], _euler_step(x, v, sig, 0))


def test_loader_reads_a_cache_written_by_the_reference(golden, tmp_path):
    """f3: the cache directory is the one the reference's own `EmbeddingCacheManager.save_cache_embedding` (data/cache_manager.py:46-93)
    wrote (stored file by file), and `CachedEmbeddingLoader` must return what the reference's `load_cache` + `pad_to_max_shape` collate
    (utils/tools.py:399-425) returned for it (values, fp16 storage), pixel `img_shapes` converted to latent-patch units."""
    from qflux_b200.cache_loader import CachedEmbeddingLoader
    c = golden["cache"]
    for rel, data in c["files"].items():
        path = tmp_path / rel
        path.parent.mkdir(parents=True, exist_ok=True)
        path.write_bytes(data)
    sizes = c["sizes"]
    ours = list(CachedEmbeddingLoader(str(tmp_path), batch_size=3, device="cpu", shuffle=False, drop_last=False))
    assert len(ours) == 1
    b = ours[0]
    for key in ("image_latents", "control_latents", "prompt_embeds"):
        assert b[key].dtype == torch.float16 and torch.equal(b[key], c["padded"][key]), key
    assert b["img_shapes"] == [[(1, H // 16, W // 16)] * 2 for H, W in sizes]
    assert b["prompt_embeds_mask"].sum(1).tolist() == [6, 11, 16]
    # ... and the same batch again from the packed shards written off that cache
    from qflux_b200.cache_loader import pack_cache
    pack_cache(str(tmp_path))
    p = list(CachedEmbeddingLoader(str(tmp_path), batch_size=3, device="cpu", shuffle=False, drop_last=False, packed=True))[0]
    assert all(torch.equal(p[k], b[k]) for k in ("image_latents", "control_latents", "prompt_embeds", "prompt_embeds_mask")) and p["img_shapes"] == b["img_shapes"]


def test_dreamomni2_trainer_rides_the_flux_kontext_path(golden):
    """§8 f4: the reference's DreamOmni2 trainer only changes what happens BEFORE the embeddings exist (VLM prompt optimisation); its loss
    recipes are FluxKontextLoraTrainer's own, i.e. exactly what FluxKontextStep / patch_trainer replace (stored: each trainer's method
    resolution order and the class defining each loss recipe)."""
    t = golden["trainers"]
    assert "FluxKontextLoraTrainer" in t["DreamOmni2Trainer"]["mro"]
    for name in ("_compute_loss", "_compute_loss_shared_mode", "_compute_loss_multi_resolution_mode"):
        assert t["DreamOmni2Trainer"]["owner"][name] == t["FluxKontextLoraTrainer"]["owner"][name] == "FluxKontextLoraTrainer", name
    # likewise BASELINE config 4's trainer: Edit-Plus only changes how the (several) control images are encoded and concatenated
    assert "QwenImageEditTrainer" in t["QwenImageEditPlusTrainer"]["mro"]
    assert t["QwenImageEditPlusTrainer"]["owner"]["_compute_loss"] == t["QwenImageEditTrainer"]["owner"]["_compute_loss"] == "QwenImageEditTrainer"


def qwen_sampling_inputs():
    """The `embeddings` dict of the Qwen validation-loop comparison (also what tests/golden/make_boundary_golden.py hands the reference)."""
    import ref_common as rc
    x = rc.rand_inputs(rc.CASES["qwen_hd128"])
    B, L = x["image_latents"].shape[:2]
    T = x["prompt_embeds"].shape[1]
    g = torch.Generator().manual_seed(77)
    return dict(num_inference_steps=4, true_cfg_scale=3.0, guidance=1.0, height=512, width=512, negative_prompt="bad",
                control_latents=x["control_latents"].bfloat16(), prompt_embeds=x["prompt_embeds"].bfloat16(),
                prompt_embeds_mask=torch.ones(B, T, dtype=torch.int64), img_shapes=x["img_shapes"],
                negative_prompt_embeds=(torch.randn(B, T - 3, x["prompt_embeds"].shape[2], generator=g) * 3).bfloat16(),
                negative_prompt_embeds_mask=torch.ones(B, T - 3, dtype=torch.int64), latents=torch.randn(B, L, 64, generator=g).bfloat16())


def flux_sampling_inputs():
    """The `embeddings` dict of the FLUX-Kontext validation-loop comparison."""
    import ref_common as rc
    from qflux_b200.train_step import FluxKontextStep
    x = rc.rand_inputs(rc.CASES["flux_hd128"])
    B, L = x["image_latents"].shape[:2]
    T, J = x["prompt_embeds"].shape[1:]
    hw = int(L ** 0.5)
    g = torch.Generator().manual_seed(78)
    return dict(num_inference_steps=4, true_cfg_scale=2.5, guidance=3.5, control_latents=x["control_latents"].bfloat16(),
                control_ids=FluxKontextStep.latent_image_ids(hw, hw, "cpu", 1.0), latent_ids=FluxKontextStep.latent_image_ids(hw, hw, "cpu", 0.0),
                latents=torch.randn(B, L, 64, generator=g).bfloat16(), pooled_prompt_embeds=x["pooled_prompt_embeds"].bfloat16(),
                prompt_embeds=x["prompt_embeds"].bfloat16(), text_ids=torch.zeros(T, 3),
                negative_pooled_prompt_embeds=torch.randn(B, x["pooled_prompt_embeds"].shape[1], generator=g).bfloat16(),
                negative_prompt_embeds=torch.randn(B, T, J, generator=g).bfloat16(), negative_text_ids=torch.zeros(T, 3))


# The stored reference-loop latents come from the emulated bf16 kernels on the CPU that generated them; CPUs with other bf16 matmul
# kernels round differently (4.9e-3 measured for the FLUX case on a second machine), so the stored comparison allows 1e-2.
ON_FUSED_TOL = 1e-2


def _rel(a, b):
    return ((a.float() - b.float()).norm() / b.float().norm()).item()


def test_reference_validation_loop_runs_on_the_fused_model(golden, emu):
    """§8 f2 pinned to the reference's own loop: `QwenImageEditTrainer.sampling_from_embeddings` (qwen_image_edit_trainer.py:1116-1289 —
    shifted schedule, `dit.cache_context`, true CFG with norm rescale, `scheduler.step`), run UNMODIFIED with `self.dit` = the fused
    model, produced the stored latents; `qflux_b200.sampler.sample_qwen` on the same model must reproduce them, and — within bf16
    tolerance — the stored latents of the same loop driving the reference's own fp32 transformer."""
    from qflux_b200 import from_reference
    from qflux_b200.sampler import sample_qwen
    fused = from_reference(_reference_module("qwen_hd128"), _host_only=True)
    emb = qwen_sampling_inputs()
    want = golden["sampling"]["qwen"]
    ours = sample_qwen(fused, dict(emb), scheduler_kwargs=dict(base_seq_len=256, max_seq_len=8192, base_shift=0.5, max_shift=0.9, shift_terminal=0.02))
    assert want["on_fused"].shape == ours.shape == emb["latents"].shape
    assert _rel(ours, want["on_fused"]) < ON_FUSED_TOL, "sampler.py must be the reference's loop"
    assert _rel(ours, want["on_reference"]) < 3e-2


def test_merge_adapter_like_peft(emu):
    """`BaseTrainer.merge_lora` -> `dit.merge_adapter()` (base_trainer.py:413-416): after merging, the adapter-free forward of the
    merged weights equals the adapted forward; `unmerge_adapter()` brings the factors back."""
    import ref_common as rc
    from qflux_b200 import from_reference
    m = from_reference(_reference_module("qwen_hd128"), _host_only=True)
    x = rc.rand_inputs(rc.CASES["qwen_hd128"])
    packed = torch.cat([x["image_latents"], x["control_latents"]], 1).bfloat16()
    kw = dict(hidden_states=packed, timestep=torch.tensor([0.5] * packed.shape[0]), encoder_hidden_states=x["prompt_embeds"].bfloat16(),
              encoder_hidden_states_mask=torch.ones(packed.shape[0], x["prompt_embeds"].shape[1], dtype=torch.int64), img_shapes=x["img_shapes"])
    with torch.no_grad():
        before = m(**kw)[0].float()
        B_norm = sum(float(p.float().norm()) for k, p in m._lora_params.items() if ".lora_B." in k)
        m.merge_adapter()
        assert all(float(p.abs().max()) == 0 for k, p in m._lora_params.items() if ".lora_B." in k) and B_norm > 0
        merged = m(**kw)[0].float()
        m.unmerge_adapter()
        after = m(**kw)[0].float()
    assert ((merged - before).norm() / before.norm()).item() < 1e-2
    assert ((after - before).norm() / before.norm()).item() < 1e-2
    assert abs(sum(float(p.float().norm()) for k, p in m._lora_params.items() if ".lora_B." in k) - B_norm) < 1e-6


def test_reference_flux_validation_loop_runs_on_the_fused_model(golden, emu):
    """The FLUX-Kontext counterpart: `FluxKontextLoraTrainer.sampling_from_embeddings` (flux_kontext_trainer.py:902-976; plain CFG, no norm
    rescale) unmodified on the fused FLUX model (stored) vs `sample_flux`, and vs the same loop on the reference's own transformer in bf16
    (an fp32 run is not comparable over several steps: a bf16 FLUX model multiplies the timestep by 1000 IN bf16,
    transformer_flux.py:707-710, so its time embedding differs from the fp32 model's at most sigmas)."""
    from qflux_b200 import from_reference
    from qflux_b200.sampler import sample_flux
    fused = from_reference(_reference_module("flux_hd128"), _host_only=True)
    emb = flux_sampling_inputs()
    want = golden["sampling"]["flux"]
    ours = sample_flux(fused, dict(emb), scheduler_kwargs=dict(base_seq_len=256, max_seq_len=4096, base_shift=0.5, max_shift=1.15))
    assert want["on_fused"].shape == ours.shape == emb["latents"].shape
    assert _rel(ours, want["on_fused"]) < ON_FUSED_TOL, "sampler.py must be the reference's loop"
    assert _rel(ours, want["on_reference"]) < 5e-2


def _accelerator():
    from accelerate import Accelerator
    acc = Accelerator()
    acc.device = torch.device("cpu")
    return acc


def test_reference_fit_setup_runs_on_the_patched_trainer(shims, emu):
    """The reference's fit-stage plumbing around the hot path, as it acts on a trainer whose `dit` is the fused model:
    `setup_model_device_train_mode("fit")` (qwen_image_edit_trainer.py:286-330: requires_grad_(False) / train() / requires_grad by
    "lora" in the name), `configure_optimizers()` (base_trainer.py:884-916: optimizer over the trainable parameters + constant schedule)
    and the DDP branch of `accelerator_prepare()` (:318-388: enable_gradient_checkpointing, AttnProcsLayers over the LoRA modules,
    accelerator.prepare, dit.to(device)); the model summary fit() logs (:634-640) walks its modules and parameters; then one loop-body
    iteration must move exactly the LoRA parameters."""
    import ref_common as rc
    from diffusers.loaders import AttnProcsLayers
    x = rc.rand_inputs(rc.CASES["qwen_hd128"])
    tr = _patched_trainer("qwen_hd128", "MseLoss")
    tr.accelerator = _accelerator()
    dit = tr.dit
    dit.requires_grad_(False)
    dit.train()
    for name, param in dit.named_parameters():
        param.requires_grad = "lora" in name
    tr.optimizer = torch.optim.AdamW([p for p in dit.parameters() if p.requires_grad], lr=1e-2, weight_decay=0.0)
    tr.lr_scheduler = torch.optim.lr_scheduler.ConstantLR(tr.optimizer, factor=1.0, total_iters=0)
    dit.enable_gradient_checkpointing()
    layers, tr.optimizer, _, tr.lr_scheduler = tr.accelerator.prepare(AttnProcsLayers(_lora_modules(dit)), tr.optimizer, [1, 2, 3],
                                                                       tr.lr_scheduler)
    assert {id(p) for p in layers.parameters()} == {id(p) for p in dit.parameters()}
    assert dit.to(tr.accelerator.device) is dit
    rows = [(n, type(mod).__name__, sum(p.numel() for p in mod.parameters())) for n, mod in dit.named_modules()]
    assert rows and rows[0][2] == sum(p.numel() for p in dit.parameters())
    names = [n for n, p in dit.named_parameters() if p.requires_grad]
    assert names and all("lora" in n for n in names) and len(names) == len(list(dit.parameters()))
    assert isinstance(tr.optimizer, torch.optim.AdamW) or isinstance(getattr(tr.optimizer, "optimizer", None), torch.optim.AdamW)
    before = {n: p.detach().clone() for n, p in dit.named_parameters()}
    e = {k: v for k, v in x.items() if k != "u"}
    with tr.accelerator.accumulate(dit):
        loss = tr._compute_loss(e)
        tr.accelerator.backward(loss)
        tr.accelerator.clip_grad_norm_(dit.parameters(), tr.config.train.max_grad_norm)
        tr.optimizer.step()
        tr.optimizer.zero_grad()
    assert torch.isfinite(loss) and all(not torch.equal(p, before[n]) for n, p in dit.named_parameters() if ".lora_A." in n)


def test_reference_train_epoch_runs_end_to_end(golden, shims, emu, tmp_path):
    """The whole inner loop as the reference ships it (`BaseTrainer.train_epoch`, base_trainer.py:508-560): per batch `training_step` ->
    `prepare_cached_embeddings` (pixel -> latent-patch img_shapes, H / (vae_scale_factor * 2)) -> the patched `_compute_loss` -> backward
    -> clip_gradients -> optimizer.step -> lr_scheduler.step -> zero_grad, fed by `CachedEmbeddingLoader(reference_batch_format=True)`
    reading a cache that the reference's `EmbeddingCacheManager` wrote (stored file by file: two samples, each twice).  The loss must be
    finite every step and go down over the epochs."""
    from qflux_b200.cache_loader import CachedEmbeddingLoader
    for rel, data in golden["epoch_cache"].items():
        path = tmp_path / rel
        path.parent.mkdir(parents=True, exist_ok=True)
        path.write_bytes(data)
    tr = _patched_trainer("qwen_hd128", "MseLoss")
    tr.accelerator = _accelerator()
    tr.config.train.max_grad_norm = 1.0
    tr.optimizer = torch.optim.AdamW([p for p in tr.dit.parameters() if p.requires_grad], lr=2e-2, weight_decay=0.0)
    tr.lr_scheduler = torch.optim.lr_scheduler.ConstantLR(tr.optimizer, factor=1.0, total_iters=0)
    px = tr.vae_scale_factor * 2
    losses = []
    torch.manual_seed(0)
    for epoch in range(6):
        for batch in CachedEmbeddingLoader(str(tmp_path), batch_size=2, device="cpu", shuffle=False, reference_batch_format=True):
            assert all(batch["cached"])
            with tr.accelerator.accumulate(tr.dit):
                batch["img_shapes"] = [[(1, H // px, W // px) for (_, H, W) in s] for s in batch["img_shapes"]]
                loss = tr._compute_loss(batch)
                tr.accelerator.backward(loss)
                tr.accelerator.clip_grad_norm_(tr.dit.parameters(), tr.config.train.max_grad_norm)
                tr.optimizer.step()
                tr.lr_scheduler.step()
                tr.optimizer.zero_grad()
            losses.append(tr.accelerator.gather(loss.detach()).mean().item())
    assert len(losses) == 12 and all(l == l and abs(l) < 1e4 for l in losses), losses
    assert sum(losses[-4:]) < sum(losses[:4]), losses
