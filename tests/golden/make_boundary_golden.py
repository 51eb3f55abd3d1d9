"""Generate tests/golden/boundary_golden.pt: what the original project's own trainer code computed in the comparisons of
tests/test_reference_trainer_boundary.py, so that those comparisons run without the original project:

    QFLUX_REFERENCE_SRC=<checkout of the original project>/src python tests/golden/make_boundary_golden.py

Stored (CPU; LoRA parameters and gradients in bf16, compared at 2e-2): the rotary tables of its `QwenEmbedRope`; the timesteps, shift and Euler update of its
`prepare_predict_timesteps`; the loss trajectory and LoRA parameters of three steps of its Qwen loop body; loss and LoRA gradients of
its FLUX-Kontext `_compute_loss` (shared and multi-resolution mode); a small embedding cache written by its `EmbeddingCacheManager`
and what its reader + `pad_to_max_shape` return for it; the latents of its Qwen and FLUX validation loops, driving the fused model
(emulated kernels) and driving its own transformer.
"""
import contextlib
import io
import os
import sys
import types

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF_SRC = os.environ["QFLUX_REFERENCE_SRC"]
for p in (ROOT, os.path.join(ROOT, "qwen-image-finetune_b200"), os.path.join(ROOT, "tests"), os.path.join(ROOT, "tests", "shims"), HERE,
          REF_SRC):
    sys.path.insert(0, p)
import stub_importer  # noqa: E402

stub_importer.install()
import make_ref_model_golden as mg  # noqa: E402
import ref_common as rc  # noqa: E402

QWEN_SCHED = dict(num_train_timesteps=1000, shift=1.0, use_dynamic_shifting=True, base_shift=0.5, max_shift=0.9, base_image_seq_len=256,
                  max_image_seq_len=8192, shift_terminal=0.02)
FLUX_SCHED = dict(num_train_timesteps=1000, shift=3.0, use_dynamic_shifting=True, base_shift=0.5, max_shift=1.15, base_image_seq_len=256,
                  max_image_seq_len=4096)
CACHE_SIZES = [(64, 64), (32, 64), (64, 48)]  # pixel (H, W) of the three cached samples


def _cfg(r=4, alpha=8, targets=("to_q", "to_k", "to_v", "to_out.0")):
    lora = types.SimpleNamespace(r=r, lora_alpha=alpha, init_lora_weights="gaussian", target_modules=list(targets), pretrained_weight=None)
    return types.SimpleNamespace(model=types.SimpleNamespace(lora=lora), train=types.SimpleNamespace(max_grad_norm=0.5, gradient_accumulation_steps=1))


def rope():
    from qflux.models.transformer_qwenimage import QwenEmbedRope
    r = QwenEmbedRope(theta=10000, axes_dim=[16, 56, 56], scale_rope=True)
    return [r([shapes], [T], device=torch.device("cpu")) for shapes, T in (([(1, 4, 4), (1, 4, 4)], 7), ([(1, 4, 6), (1, 4, 6), (1, 2, 8)], 11))]


def schedule():
    from diffusers.schedulers.scheduling_flow_match_euler_discrete import FlowMatchEulerDiscreteScheduler
    from qflux.trainer.base_trainer import BaseTrainer
    from qflux.utils.sampling import calculate_shift
    out, g = [], torch.Generator().manual_seed(9)
    for conf in (QWEN_SCHED, FLUX_SCHED):
        for steps, seq in ((20, 1024), (8, 4096), (50, 400)):
            tr = types.SimpleNamespace(sampling_scheduler=FlowMatchEulerDiscreteScheduler(**conf), scheduler=None, dit=torch.nn.Linear(1, 1))
            with contextlib.redirect_stdout(io.StringIO()):
                ts, n = BaseTrainer.prepare_predict_timesteps(tr, steps, seq)
            shift = calculate_shift(seq, conf["base_image_seq_len"], conf["max_image_seq_len"], conf["base_shift"], conf["max_shift"])
            x, v = torch.randn(2, 8, 64, generator=g).bfloat16(), torch.randn(2, 8, 64, generator=g).bfloat16()
            tr.sampling_scheduler.set_begin_index(0)
            step = tr.sampling_scheduler.step(v, ts[0], x, return_dict=False)[0]
            out.append(dict(steps=steps, seq=seq, timesteps=ts.cpu(), n=n, shift=shift, sigmas=tr.sampling_scheduler.sigmas.cpu(),
                            euler_step=step))  # x, v: drawn again from the same seeded generator by the test
    return out


def loop_body():
    """Three iterations of base_trainer.py:518-533 on the un-patched trainer (the reference model, fp32)."""
    from qflux.losses import MseLoss
    from qflux.trainer.qwen_image_edit_trainer import QwenImageEditTrainer
    import qflux.trainer.qwen_image_edit_trainer as qt
    spec = rc.CASES["qwen_hd128"]
    x = rc.rand_inputs(spec)
    emb = {k: v for k, v in x.items() if k != "u"}
    orig = qt.compute_density_for_timestep_sampling
    qt.compute_density_for_timestep_sampling = lambda **kw: x["u"].clone()
    try:
        dit, _ = mg.build_reference(spec)
        tr = mg._trainer(QwenImageEditTrainer, dit, MseLoss(reduction="mean"))
        tr.config = _cfg()
        tr.adapter_name = "default"
        tr.optimizer = torch.optim.AdamW([p for p in tr.dit.parameters() if p.requires_grad], lr=1e-2, weight_decay=0.0)
        losses = []
        for it in range(3):
            with tr.accelerator.accumulate(tr.dit):
                torch.manual_seed(100 + it)
                loss = tr._compute_loss(dict(emb))
                tr.accelerator.backward(loss)
                tr.clip_gradients()
                tr.optimizer.step()
                tr.optimizer.zero_grad()
            losses.append(loss.item())
    finally:
        qt.compute_density_for_timestep_sampling = orig
    # bf16 storage (relative rounding 4e-3) against a 2e-2 tolerance
    return dict(losses=losses, params={n: p.detach().bfloat16() for n, p in tr.dit.named_parameters() if p.requires_grad})


def flux_train():
    from qflux.losses import AttentionMaskMseLoss, MseLoss
    from qflux.trainer.flux_kontext_trainer import FluxKontextLoraTrainer
    out = {}
    for case, crit in (("flux_hd128", MseLoss(reduction="mean")), ("flux_custom_multires", AttentionMaskMseLoss(reduction="mean"))):
        spec = rc.CASES[case]
        x = rc.rand_inputs(spec)
        emb = {k: v for k, v in x.items() if k not in ("img_shapes_latent", "hw")}
        if spec["kind"] == "flux":
            h_, w_ = x["hw"]
            emb["control_ids"] = FluxKontextLoraTrainer._prepare_latent_image_ids(1, h_, w_, torch.device("cpu"), torch.float32)
            emb["control_ids"][..., 0] = 1
            emb["img_shapes"] = [[(3, h_ * 16, w_ * 16), (3, h_ * 16, w_ * 16)]] * spec["B"]
        else:
            emb["timestep"] = x["timestep"].view(-1, 1)
        dit, _ = mg.build_reference(spec)
        tr = mg._trainer(FluxKontextLoraTrainer, dit, crit)
        tr.config = _cfg()
        loss = tr._compute_loss(dict(emb))
        loss.backward()
        out[case] = dict(control_ids=emb.get("control_ids"), loss=loss.item(),
                         grads={n: p.grad.bfloat16() for n, p in tr.dit.named_parameters() if p.requires_grad and p.grad is not None})
    return out


def cache(tmp):
    from qflux.data.cache_manager import EmbeddingCacheManager
    from qflux.utils.tools import pad_to_max_shape
    mgr = EmbeddingCacheManager(tmp)
    g = torch.Generator().manual_seed(5)
    hashes = []
    for i, (H, W) in enumerate(CACHE_SIZES):
        L, T = (H // 16) * (W // 16), 6 + 5 * i
        data = dict(image_latents=torch.randn(L, 64, generator=g), control_latents=torch.randn(L, 64, generator=g),
                    prompt_embeds=torch.randn(T, 48, generator=g))
        fh = dict(main_hash=f"m{i:03d}", image_hash=f"i{i:03d}", control_hash=f"c{i:03d}", prompt_hash=f"p{i:03d}")
        mgr.save_cache_embedding(data, dict(image_latents="image_hash", control_latents="control_hash", prompt_embeds="prompt_hash"), fh,
                                 img_shapes=[[3, H, W], [3, H, W]])
        hashes.append(fh)
    files = _files(tmp)
    theirs = [mgr.load_cache({"file_hashes": fh}) for fh in hashes]
    padded = {k: pad_to_max_shape([t[k] for t in theirs]) for k in ("image_latents", "control_latents", "prompt_embeds")}
    return dict(sizes=CACHE_SIZES, files=files, padded=padded)


def sampling():
    import emu_lib
    from diffusers.schedulers.scheduling_flow_match_euler_discrete import FlowMatchEulerDiscreteScheduler
    from qflux.trainer.base_trainer import BaseTrainer
    from qflux.trainer.flux_kontext_trainer import FluxKontextLoraTrainer
    from qflux.trainer.qwen_image_edit_trainer import QwenImageEditTrainer
    from qflux_b200 import from_reference, lib
    from test_reference_trainer_boundary import flux_sampling_inputs, qwen_sampling_inputs
    restore = emu_lib.install(lib)
    out = {}
    try:
        for kind, cls, sched, make in (("qwen", QwenImageEditTrainer, QWEN_SCHED, qwen_sampling_inputs),
                                       ("flux", FluxKontextLoraTrainer, FLUX_SCHED, flux_sampling_inputs)):
            ref_dit, _ = mg.build_reference(rc.CASES[f"{kind}_hd128"])
            fused = from_reference(ref_dit, _host_only=True)
            emb = make()

            def loop(dit, dtype):
                tr = types.SimpleNamespace(dit=dit, vae_scale_factor=8, weight_dtype=dtype, scheduler=None,
                                           sampling_scheduler=FlowMatchEulerDiscreteScheduler(**sched))
                tr.prepare_predict_timesteps = lambda *a, **k: BaseTrainer.prepare_predict_timesteps(tr, *a, **k)
                with contextlib.redirect_stdout(io.StringIO()), contextlib.redirect_stderr(io.StringIO()):
                    return cls.sampling_from_embeddings(tr, dict(emb)).float()
            # the reference's own transformer: fp32 for Qwen; bf16 for FLUX (its bf16 model multiplies the timestep by 1000 IN bf16,
            # transformer_flux.py:707-710, so an fp32 run is not comparable over several steps)
            own = loop(ref_dit.float(), torch.float32) if kind == "qwen" else loop(ref_dit.bfloat16(), torch.bfloat16)
            out[kind] = dict(on_fused=loop(fused, torch.bfloat16), on_reference=own)
    finally:
        restore()
    return out


def save_lora(tmp):
    """The safetensors header of the file its `save_lora` writes for the fused model (the tensor values are the model's LoRA factors,
    filled by name), what its `classify_lora_weight` calls that file, and the LoRA parameter names its own transformer has after
    loading it through `load_lora_adapter`."""
    import json
    import struct
    from accelerate import Accelerator
    from diffusers import FluxKontextPipeline
    from qflux.models.transformer_qwenimage import QwenImageTransformer2DModel
    from qflux.trainer.base_trainer import BaseTrainer
    from qflux.trainer.qwen_image_edit_trainer import QwenImageEditTrainer
    from qflux.utils.lora_utils import classify_lora_weight
    from test_reference_trainer_boundary import _cfg as test_cfg
    from test_reference_trainer_boundary import _fused
    m = _fused()
    BaseTrainer.add_lora_adapter(m, test_cfg(), "default")
    rc.det_fill_(type("B", (), {"named_parameters": lambda s: iter(m._lora_params.items())})(), 5)
    tr = object.__new__(QwenImageEditTrainer)
    tr.accelerator, tr.dit, tr.adapter_name, tr.pipeline_class = Accelerator(), m, "default", FluxKontextPipeline
    tr.save_lora(os.path.join(tmp, "ckpt"))
    path = os.path.join(tmp, "ckpt", "pytorch_lora_weights.safetensors")
    with open(path, "rb") as f:
        n = struct.unpack("<Q", f.read(8))[0]
        header = json.loads(f.read(n))
    with contextlib.redirect_stdout(io.StringIO()):
        refm = QwenImageTransformer2DModel(**rc.QWEN_HD128)
    refm.load_lora_adapter(path, adapter_name="default")
    return dict(header=header, kind=classify_lora_weight(path), reference_lora_names=sorted(n for n, _ in refm.named_parameters() if "lora_" in n))


def trainer_facts():
    """For each trainer class: its method resolution order and which class defines each loss recipe."""
    from qflux.trainer.dreamomni2_trainer import DreamOmni2Trainer
    from qflux.trainer.flux_kontext_trainer import FluxKontextLoraTrainer
    from qflux.trainer.qwen_image_edit_plus_trainer import QwenImageEditPlusTrainer
    from qflux.trainer.qwen_image_edit_trainer import QwenImageEditTrainer
    out = {}
    for cls in (DreamOmni2Trainer, FluxKontextLoraTrainer, QwenImageEditPlusTrainer, QwenImageEditTrainer):
        owner = {name: next((k.__name__ for k in cls.__mro__ if name in vars(k)), None)
                 for name in ("_compute_loss", "_compute_loss_shared_mode", "_compute_loss_multi_resolution_mode")}
        out[cls.__name__] = dict(mro=[k.__name__ for k in cls.__mro__], owner=owner)
    return out


def epoch_cache(tmp):
    """The cache its `EmbeddingCacheManager` writes for the train_epoch test: two samples, each stored twice."""
    from qflux.data.cache_manager import EmbeddingCacheManager
    mgr, J = EmbeddingCacheManager(tmp), rc.QWEN_HD128["joint_attention_dim"]
    for i in range(4):
        gi = torch.Generator().manual_seed(40 + i % 2)
        data = dict(image_latents=torch.randn(16, 64, generator=gi), control_latents=torch.randn(16, 64, generator=gi),
                    prompt_embeds=torch.randn(6, J, generator=gi) * 3)
        fh = dict(main_hash=f"m{i}", image_hash=f"i{i}", control_hash=f"c{i}", prompt_hash=f"p{i}")
        mgr.save_cache_embedding(data, dict(image_latents="image_hash", control_latents="control_hash", prompt_embeds="prompt_hash"), fh,
                                 img_shapes=[[3, 64, 64], [3, 64, 64]])
    return _files(tmp)


def _files(root):
    files = {}
    for d, _, names in os.walk(root):
        for n in names:
            with open(os.path.join(d, n), "rb") as f:
                files[os.path.relpath(os.path.join(d, n), root)] = f.read()
    return files


def _compact(o):
    """torch.save writes a view's whole storage (the rotary tables are slices of a cached table): store compact copies."""
    if torch.is_tensor(o):
        return o.detach().clone()
    if isinstance(o, dict):
        return {k: _compact(v) for k, v in o.items()}
    if isinstance(o, (list, tuple)):
        return type(o)(_compact(v) for v in o)
    return o


def main():
    import tempfile
    with tempfile.TemporaryDirectory() as tmp:
        out = dict(rope=rope(), schedule=schedule(), loop_body=loop_body(), flux_train=flux_train(), cache=cache(tmp), sampling=sampling())
    with tempfile.TemporaryDirectory() as tmp:
        out["save_lora"] = save_lora(tmp)
    with tempfile.TemporaryDirectory() as tmp:
        out["epoch_cache"] = epoch_cache(tmp)
    out["trainers"] = trainer_facts()
    path = os.path.join(HERE, "boundary_golden.pt")
    torch.save(_compact(out), path)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    main()
