"""Generate tests/golden/* by RUNNING THE REAL REFERENCE (/root/reference/lora_diffusion/lora.py
and cli_svd.py, loaded by file path because the package import needs fire/diffusers) on small
seeded inputs. Run in the build container (the reference tree does not exist on the GPU box):

    python scripts/make_golden.py

Outputs (all small, committed):
  golden/ops_linear.pt, ops_conv.pt     operator forward + autograd grads (fp32, CPU)
  golden/ctor_rng.pt                    lora_down init values after manual_seed(0) (RNG parity)
  golden/inject_tiny.json               site names/order from the reference's inject on the tiny
                                        host UNet / CLIP (default + extended target sets)
  golden/tiny_saved.safetensors         save_safeloras output of the reference on the tiny models
  golden/example_loras_manifest.json    keys / shapes / dtypes / metadata / sha256 of the ten
                                        fixture files in /root/reference/example_loras
  golden/svd_distill.pt                 cli_svd.overwrite_base outputs on small matrices
  golden/adamw_clip.pt                  clip_grad_norm_ + torch.optim.AdamW trajectories
  golden/pti_loss_step.pt               cli_lora_pti.loss_step losses (plain / t_mult / masked / inpainting)
  golden/ti_train_inversion.pt          cli_lora_pti.train_inversion: 3 real steps (grads, lr, rows after)
  golden/pti_perform_tuning.pt          cli_lora_pti.perform_tuning: 3 real steps (losses, lrs, all factors after)
  golden/reference_live.json            namespace, signatures and tiny-model outputs of lora.py (digests)
  golden/reference_modules_fp32.pt      the operator classes' fp32 forward + backward on small inputs
  golden/reference_formats.json         lora_join, cli_lora_add.add, to_ckpt_v2 key conversion (digests)

    python scripts/make_golden.py live formats        (only the named generators)
"""
import hashlib
import importlib.util
import itertools
import json
import os
import sys
import types

import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
REF = "/root/reference"
OUT = os.path.join(ROOT, "tests", "golden")
os.makedirs(OUT, exist_ok=True)


def load_ref_lora():
    spec = importlib.util.spec_from_file_location("ref_lora", f"{REF}/lora_diffusion/lora.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def load_ref_svd(ref_lora):
    """cli_svd.py imports fire and diffusers at module top; stub them, and satisfy its relative
    import `.lora` with the already-loaded reference module."""
    pkg = types.ModuleType("lora_diffusion_ref")
    pkg.__path__ = [f"{REF}/lora_diffusion"]
    sys.modules["lora_diffusion_ref"] = pkg
    sys.modules["lora_diffusion_ref.lora"] = ref_lora
    sys.modules.setdefault("fire", types.ModuleType("fire"))
    d = types.ModuleType("diffusers")
    d.StableDiffusionPipeline = object
    sys.modules.setdefault("diffusers", d)
    spec = importlib.util.spec_from_file_location("lora_diffusion_ref.cli_svd", f"{REF}/lora_diffusion/cli_svd.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def gen_ops(R):
    cases = []
    for i, (M, K, N, r, bias, scale, diag) in enumerate([
            (24, 16, 24, 4, True, 1.0, False), (10, 32, 8, 1, False, 0.5, False),
            (33, 40, 48, 8, True, 1.7, True), (7, 64, 64, 16, True, 0.25, True)]):
        torch.manual_seed(100 + i)
        m = R.LoraInjectedLinear(K, N, bias, r=r, dropout_p=0.0, scale=scale)
        m.lora_up.weight.data.normal_(0, 0.1)
        d = None
        if diag:
            d = torch.rand(r) + 0.5
            m.set_selector_from_diag(d)
        x = torch.randn(2, M, K, requires_grad=True)
        y = m(x)
        gy = torch.randn_like(y)
        y.backward(gy)
        cases.append(dict(x=x.detach(), W=m.linear.weight.detach(), b=None if not bias else m.linear.bias.detach(),
                          A=m.lora_down.weight.detach(), B=m.lora_up.weight.detach(), scale=scale, diag=d,
                          y=y.detach(), gy=gy, dX=x.grad, dA=m.lora_down.weight.grad, dB=m.lora_up.weight.grad,
                          dW_is_none=True))
    torch.save(cases, f"{OUT}/ops_linear.pt")

    conv = []
    for i, (Cin, Cout, k, pad, r, bias, scale, HW) in enumerate([
            (8, 16, 3, 1, 4, True, 1.0, 6), (16, 8, 1, 0, 4, False, 0.5, 5), (12, 12, 3, 1, 8, True, 2.0, 9)]):
        torch.manual_seed(200 + i)
        m = R.LoraInjectedConv2d(Cin, Cout, k, 1, pad, 1, 1, bias, r=r, dropout_p=0.0, scale=scale)
        m.lora_up.weight.data.normal_(0, 0.1)
        x = torch.randn(2, Cin, HW, HW, requires_grad=True)
        y = m(x)
        gy = torch.randn_like(y)
        y.backward(gy)
        conv.append(dict(x=x.detach(), W=m.conv.weight.detach(), b=None if not bias else m.conv.bias.detach(),
                         A=m.lora_down.weight.detach(), B=m.lora_up.weight.detach(), scale=scale, padding=pad,
                         y=y.detach(), gy=gy, dX=x.grad, dA=m.lora_down.weight.grad, dB=m.lora_up.weight.grad))
    torch.save(conv, f"{OUT}/ops_conv.pt")

    # dropout statistics are not golden-able (Philox stream); keep the p>0 eval-mode identity
    torch.manual_seed(7)
    m = R.LoraInjectedLinear(16, 16, False, r=4, dropout_p=0.1)
    m.lora_up.weight.data.normal_(0, 0.1)
    m.eval()
    x = torch.randn(5, 16)
    torch.save(dict(x=x, W=m.linear.weight.detach(), A=m.lora_down.weight.detach(), B=m.lora_up.weight.detach(),
                    y_eval=m(x).detach()), f"{OUT}/ops_dropout_eval.pt")


def gen_ctor_rng(R):
    out = {}
    torch.manual_seed(0)
    m = R.LoraInjectedLinear(16, 24, True, r=4)
    out["linear_down"] = m.lora_down.weight.detach().clone()
    out["linear_next_rand"] = torch.rand(3)
    torch.manual_seed(0)
    c = R.LoraInjectedConv2d(8, 12, 3, 1, 1, r=4)
    out["conv_down"] = c.lora_down.weight.detach().clone()
    out["conv_next_rand"] = torch.rand(3)
    torch.save(out, f"{OUT}/ctor_rng.pt")


def gen_inject(R):
    from lora_b200.host.clip import build_text_encoder
    from lora_b200.host.unet_sd15 import UNet2DConditionModel, UNetConfig
    res = {}
    torch.manual_seed(0)
    unet = UNet2DConditionModel(UNetConfig.tiny())
    _, names = R.inject_trainable_lora(unet, r=4)
    res["unet_default_names"] = names
    res["unet_default_shapes"] = [[list(m.lora_up.weight.shape), list(m.lora_down.weight.shape)]
                                  for m in unet.modules() if m.__class__.__name__.startswith("LoraInjected")]
    torch.manual_seed(0)
    unet2 = UNet2DConditionModel(UNetConfig.tiny())
    _, names2 = R.inject_trainable_lora_extended(unet2, r=4)
    res["unet_extended_names"] = names2
    res["unet_extended_kinds"] = [m.__class__.__name__ for m in unet2.modules()
                                  if m.__class__.__name__.startswith("LoraInjected")]
    res["unet_extended_shapes"] = [[list(m.lora_up.weight.shape), list(m.lora_down.weight.shape)]
                                   for m in unet2.modules() if m.__class__.__name__.startswith("LoraInjected")]
    torch.manual_seed(0)
    te = build_text_encoder(tiny=True)
    _, names3 = R.inject_trainable_lora(te, target_replace_module={"CLIPAttention"}, r=4)
    res["text_names"] = names3
    # a saved file from the reference, with non-trivial factors and scale
    g = torch.Generator().manual_seed(5)
    for mdl in (unet, te):
        for m in mdl.modules():
            if m.__class__.__name__ == "LoraInjectedLinear":
                m.lora_up.weight.data.normal_(0, 0.05, generator=g)
    R.tune_lora_scale(unet, 0.5)
    R.save_safeloras_with_embeds({"unet": (unet, R.DEFAULT_TARGET_REPLACE),
                                  "text_encoder": (te, R.TEXT_ENCODER_DEFAULT_TARGET_REPLACE)},
                                 {"<s1>": torch.arange(48, dtype=torch.float32)},
                                 f"{OUT}/tiny_saved.safetensors")
    # the raw factors that produced it (so the test can rebuild the same state with our API)
    raw = {"unet": [], "text_encoder": []}
    for key, mdl in (("unet", unet), ("text_encoder", te)):
        for m in mdl.modules():
            if m.__class__.__name__ == "LoraInjectedLinear":
                raw[key].append((m.lora_up.weight.detach().clone(), m.lora_down.weight.detach().clone()))
    torch.save(raw, f"{OUT}/tiny_saved_raw.pt")
    json.dump(res, open(f"{OUT}/inject_tiny.json", "w"), indent=1)


def gen_manifest(R):
    from safetensors import safe_open
    man = {}
    d = f"{REF}/example_loras"
    for fn in sorted(os.listdir(d)):
        if not fn.endswith(".safetensors"):
            continue
        f = safe_open(f"{d}/{fn}", framework="pt", device="cpu")
        ent = {"metadata": f.metadata(), "tensors": {}}
        for k in sorted(f.keys()):
            t = f.get_tensor(k)
            ent["tensors"][k] = [list(t.shape), str(t.dtype).replace("torch.", ""),
                                 hashlib.sha256(t.contiguous().view(torch.uint8).numpy().tobytes()).hexdigest()[:16]]
        parsed = R.parse_safeloras(f)
        ent["parsed"] = {name: {"n_weights": len(w), "ranks": r, "targets": sorted(t)}
                         for name, (w, r, t) in parsed.items()}
        ent["embeds"] = sorted(R.parse_safeloras_embeds(f).keys())
        man[fn] = ent
    json.dump(man, open(f"{OUT}/example_loras_manifest.json", "w"))


def gen_svd(R):
    S = load_ref_svd(R)
    out = []
    for i, (N, K, rank, conv) in enumerate([(48, 32, 4, False), (24, 64, 8, False), (16, 8, 4, True)]):
        torch.manual_seed(300 + i)

        class Holder(nn.Module):
            def __init__(self):
                super().__init__()
                if conv:
                    self.m = R.LoraInjectedConv2d(K, N, 3, 1, 1, r=rank)
                else:
                    self.m = R.LoraInjectedLinear(K, N, False, r=rank)

            @property
            def device(self):
                return torch.device("cpu")

            @property
            def dtype(self):
                return torch.float32

        base, tuned = Holder(), Holder()
        wb = (base.m.conv if conv else base.m.linear).weight
        wt = (tuned.m.conv if conv else tuned.m.linear).weight
        low = torch.randn(N, rank) @ torch.randn(rank, wb[0].numel()) * 0.02
        wt.data = wb.data + low.reshape(wb.shape) + torch.randn_like(wb) * 1e-3
        S.overwrite_base(base, tuned, rank=rank, clamp_quantile=0.99)
        out.append(dict(Wb=wb.detach().clone(), Wt=wt.detach().clone(), rank=rank, conv=conv, q=0.99,
                        up=base.m.lora_up.weight.detach().clone(), down=base.m.lora_down.weight.detach().clone()))
    torch.save(out, f"{OUT}/svd_distill.pt")


def gen_adamw():
    torch.manual_seed(400)
    ps = [torch.randn(6, 4), torch.randn(4, 10), torch.randn(3, 3)]
    lrs = [1e-3, 1e-3, 5e-4]
    twins = [p.clone().requires_grad_(True) for p in ps]
    opt = torch.optim.AdamW([{"params": twins[:2], "lr": 1e-3}, {"params": twins[2:], "lr": 5e-4}],
                            betas=(0.9, 0.999), weight_decay=1e-2, eps=1e-8)
    traj = []
    for step in range(1, 5):
        gs = [torch.randn_like(p) * (2.0 if step % 2 else 0.05) for p in ps]
        for t, g in zip(twins, gs):
            t.grad = g.clone()
        total = torch.nn.utils.clip_grad_norm_(twins, 1.0)
        opt.step()
        traj.append(dict(grads=gs, total_norm=float(total), params=[t.detach().clone() for t in twins]))
    torch.save(dict(p0=ps, lrs=lrs, traj=traj), f"{OUT}/adamw_clip.pt")


def load_ref_pti(ref_lora):
    """cli_lora_pti.py pulls diffusers / fire / the lora_diffusion package at module top; none of
    them is touched by `loss_step` itself. Stand-ins whose attributes are inert placeholders let the
    real file execute so that the real function object can be called."""
    class _Inert(types.ModuleType):
        def __getattr__(self, name):
            if name.startswith("__"):
                raise AttributeError(name)
            return type(name, (), {"__init__": lambda self, *a, **k: None})
    saved = {}
    # huggingface_hub is installed but no longer has the names the file asks for: shadow it too
    for name in ("fire", "diffusers", "diffusers.optimization", "lora_diffusion", "wandb", "huggingface_hub"):
        saved[name] = sys.modules.get(name)
        sys.modules[name] = _Inert(name)
    try:
        spec = importlib.util.spec_from_file_location("ref_cli_lora_pti", f"{REF}/lora_diffusion/cli_lora_pti.py")
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        for name, old in saved.items():
            if old is None:
                sys.modules.pop(name, None)
            else:
                sys.modules[name] = old
    return mod


def gen_loss_step(R):
    """The PTI/Dreambooth loss of one step, computed by the reference's own `loss_step`
    (cli_lora_pti.py:260-370) on the tiny host models, CPU fp32, cached latents: plain, t_mutliplier
    0.8, masked loss (two temperatures), inpainting (9-channel input), inpainting + mask."""
    from lora_b200.host.clip import build_text_encoder
    from lora_b200.host.ddpm import DDPMNoiser
    from lora_b200.host.unet_sd15 import UNet2DConditionModel, UNetConfig
    P = load_ref_pti(R)
    noiser = DDPMNoiser(device="cpu")

    class Sched:                      # what loss_step reads from a diffusers DDPMScheduler
        config = types.SimpleNamespace(num_train_timesteps=noiser.num_train_timesteps, prediction_type="epsilon")
        add_noise = staticmethod(noiser.add_noise)

    g = torch.Generator().manual_seed(77)
    lat = torch.randn(2, 4, 8, 8, generator=g) * 0.18215
    ids = torch.randint(0, 1000, (2, 77), generator=g)
    loss_mask = (torch.rand(2, 1, 64, 64, generator=g) > 0.4).float()          # image resolution
    inp_mask = (torch.rand(2, 1, 8, 8, generator=g) > 0.5).float()             # cached: latent resolution
    inp_lat = torch.randn(2, 4, 8, 8, generator=g) * 0.18215
    cases = []
    for name, in_ch, kw, with_mask in [
            ("plain", 4, dict(), False),
            ("t_mult_0.8", 4, dict(t_mutliplier=0.8), False),
            ("masked_T1", 4, dict(mask_temperature=1.0), True),
            ("masked_T2.5", 4, dict(mask_temperature=2.5), True),
            ("inpaint", 9, dict(train_inpainting=True), False),
            ("inpaint_masked", 9, dict(train_inpainting=True, mask_temperature=1.0), True)]:
        torch.manual_seed(0)
        cfg = UNetConfig.tiny()
        cfg.in_channels = in_ch
        unet = UNet2DConditionModel(cfg)
        text = build_text_encoder(tiny=True)
        # a live LoRA branch (reference modules, non-zero up) so that the loss depends on it
        R.inject_trainable_lora(unet, r=4)
        gg = torch.Generator().manual_seed(5)
        for m in unet.modules():
            if type(m).__name__ == "LoraInjectedLinear":
                m.lora_down.weight.data.normal_(0, 0.25, generator=gg)     # explicit: independent of ctor RNG
                m.lora_up.weight.data.normal_(0, 0.05, generator=gg)
                m.dropout.p = 0.0
        batch = {"pixel_values": lat, "input_ids": ids}
        if in_ch == 9:
            batch.update(masked_image_latents=inp_lat, mask_values=inp_mask)
        if with_mask:
            batch["mask"] = loss_mask
        text.train(False), unet.train(False)
        torch.manual_seed(1234)
        loss = P.loss_step(batch, unet, None, text, Sched, cached_latents=True, **kw)
        cases.append(dict(name=name, in_channels=in_ch, kwargs=kw, with_mask=with_mask, loss=float(loss)))
    torch.save(dict(latents=lat, input_ids=ids, loss_mask=loss_mask, inpaint_mask=inp_mask,
                    masked_latents=inp_lat, model_seed=0, up_seed=5, step_seed=1234, cases=cases),
               f"{OUT}/pti_loss_step.pt")
    print({c["name"]: c["loss"] for c in cases})


def gen_ti(R):
    """Textual-inversion phase: the reference's own `train_inversion` loop (cli_lora_pti.py:373-542)
    run for 3 steps on the tiny models, CPU fp32, with torch.optim.AdamW over the embedding table
    built as at :889-895 and a LambdaLR warm-up so that the learning rate (and the norm-decay
    lambda that follows it, :456) changes every step. Recorded: per step the gradient rows of the
    placeholder tokens, the lr in force, and the placeholder rows + whole-table sum afterwards."""
    from lora_b200.host.clip import build_text_encoder
    from lora_b200.host.ddpm import DDPMNoiser
    from lora_b200.host.unet_sd15 import UNet2DConditionModel, UNetConfig
    P = load_ref_pti(R)
    noiser = DDPMNoiser(device="cpu")

    class Sched:
        config = types.SimpleNamespace(num_train_timesteps=noiser.num_train_timesteps, prediction_type="epsilon")
        add_noise = staticmethod(noiser.add_noise)

    torch.manual_seed(0)
    unet = UNet2DConditionModel(UNetConfig.tiny())
    text = build_text_encoder(tiny=True)
    unet.requires_grad_(False)
    for prm in itertools.chain(text.text_model.encoder.parameters(), text.text_model.final_layer_norm.parameters(),
                               text.text_model.embeddings.position_embedding.parameters()):
        prm.requires_grad = False
    emb = text.get_input_embeddings()
    V, D = emb.weight.shape
    tok = [V - 2, V - 1]
    index_no_updates = torch.arange(V) != -1
    for t in tok:
        index_no_updates[t] = False
    g = torch.Generator().manual_seed(21)
    batches = []
    for _ in range(3):
        ids = torch.randint(0, V - 2, (2, 77), generator=g)
        ids[0, 5], ids[1, 9], ids[1, 10] = tok[0], tok[1], tok[0]
        batches.append({"pixel_values": torch.randn(2, 4, 8, 8, generator=g) * 0.18215, "input_ids": ids})
    base_lr, wd = 5e-3, 1e-2
    steps = []

    class Recording(torch.optim.AdamW):
        def step(self, closure=None):
            steps.append(dict(grad_rows=emb.weight.grad[tok].detach().clone(), lr=self.param_groups[0]["lr"]))
            return super().step(closure)

    opt = Recording(emb.parameters(), lr=base_lr, betas=(0.9, 0.999), eps=1e-08, weight_decay=wd)
    sched = torch.optim.lr_scheduler.LambdaLR(opt, lambda k: min(1.0, (k + 1) / 4))

    class Snap:                     # lr_scheduler as train_inversion uses it; snapshots the table it finds
        def step(self_inner):
            if steps:
                steps[-1].update(rows_after=emb.weight.data[tok].clone(), table_sum=float(emb.weight.data.double().sum()))
            sched.step()

        def get_last_lr(self_inner):
            return sched.get_last_lr()

    table0_rows = emb.weight.data[tok].clone()
    table0_sum = float(emb.weight.data.double().sum())
    torch.manual_seed(4321)
    import contextlib, io
    with contextlib.redirect_stdout(io.StringIO()):
        P.train_inversion(unet, None, text, batches, 3, Sched, index_no_updates, opt, 10 ** 9, tok, ["<a>", "<b>"],
                          "/nonexistent", None, Snap(), "/nonexistent", True, clip_ti_decay=True)
    steps[-1].update(rows_after=emb.weight.data[tok].clone(), table_sum=float(emb.weight.data.double().sum()))
    assert len(steps) == 3 and all("rows_after" in s for s in steps)
    torch.save(dict(model_seed=0, token_ids=tok, base_lr=base_lr, weight_decay=wd, table0_rows=table0_rows,
                    table0_sum=table0_sum, steps=steps), f"{OUT}/ti_train_inversion.pt")
    print("ti lrs", [s["lr"] for s in steps], "row norms", [s["rows_after"].norm(dim=-1).tolist() for s in steps])


def gen_tuning(R):
    """LoRA-tuning phase: the reference's own `perform_tuning` loop (cli_lora_pti.py:545-680) for 3
    steps, CPU fp32 (its `torch.cuda.amp.autocast()` is inert without CUDA), on the tiny UNet + text
    encoder injected by the reference's `inject_trainable_lora` (r=4), AdamW param groups built as
    at :958-997 (unet_lr 1e-4 / text_encoder_lr 1e-5, weight_decay_lora 1e-3), a LambdaLR linear
    decay. Every factor is set from a seeded generator first, so the trajectory depends on no
    constructor RNG. Recorded: per-step loss and lr, and every factor after the 3 steps."""
    from lora_b200.host.clip import build_text_encoder
    from lora_b200.host.ddpm import DDPMNoiser
    from lora_b200.host.unet_sd15 import UNet2DConditionModel, UNetConfig
    P = load_ref_pti(R)
    noiser = DDPMNoiser(device="cpu")

    class Sched:
        config = types.SimpleNamespace(num_train_timesteps=noiser.num_train_timesteps, prediction_type="epsilon")
        add_noise = staticmethod(noiser.add_noise)

    torch.manual_seed(0)
    unet = UNet2DConditionModel(UNetConfig.tiny())
    text = build_text_encoder(tiny=True)
    unet.requires_grad_(False)
    text.requires_grad_(False)
    up, _ = R.inject_trainable_lora(unet, r=4)
    tp, _ = R.inject_trainable_lora(text, target_replace_module={"CLIPAttention"}, r=4)
    gg = torch.Generator().manual_seed(6)
    sites = [m for m in list(unet.modules()) + list(text.modules()) if type(m).__name__ == "LoraInjectedLinear"]
    for m in sites:
        m.lora_down.weight.data.normal_(0, 0.25, generator=gg)
        m.lora_up.weight.data.normal_(0, 0.05, generator=gg)
    opt = torch.optim.AdamW([{"params": itertools.chain(*up), "lr": 1e-4},
                             {"params": itertools.chain(*tp), "lr": 1e-5}], weight_decay=1e-3)
    sched = torch.optim.lr_scheduler.LambdaLR(opt, lambda k: max(0.0, 1.0 - k / 6))
    g = torch.Generator().manual_seed(22)
    V = text.get_input_embeddings().weight.shape[0]
    batches = [{"pixel_values": torch.randn(2, 4, 8, 8, generator=g) * 0.18215,
                "input_ids": torch.randint(0, V, (2, 77), generator=g),
                "mask": (torch.rand(2, 1, 64, 64, generator=g) > 0.4).float()} for _ in range(3)]
    rec = []

    class Recording:
        def step(self_inner):
            sched.step()
            rec.append(dict(lrs=[grp["lr"] for grp in opt.param_groups]))

        def get_last_lr(self_inner):
            return sched.get_last_lr()

    real_loss_step = P.loss_step

    def spy(*a, **k):
        out = real_loss_step(*a, **k)
        rec[-1]["loss"] = float(out.detach())
        rec[-1]["kwargs"] = {kk: vv for kk, vv in k.items() if isinstance(vv, (int, float, bool))}
        return out

    P.loss_step = spy
    torch.manual_seed(999)
    import contextlib, io
    try:
        with contextlib.redirect_stdout(io.StringIO()):
            P.perform_tuning(unet, None, text, batches, 3, Sched, opt, 10 ** 9, [], [], "/nonexistent",
                             Recording(), {"CrossAttention", "Attention", "GEGLU"}, {"CLIPAttention"}, 1.0,
                             "out", None, "/nonexistent", True)
    finally:
        P.loss_step = real_loss_step
    assert len(rec) == 3 and rec[0]["kwargs"]["t_mutliplier"] == 0.8
    keep = sorted({0, 1, 2, len(up) // 2 - 1, len(up) // 2, len(sites) - 1})      # a few sites in full ...
    factors = {i: (sites[i].lora_up.weight.detach().clone(), sites[i].lora_down.weight.detach().clone()) for i in keep}
    sums = [(float(m.lora_up.weight.double().sum()), float(m.lora_down.weight.double().sum()),     # ... all by moments
             float((m.lora_up.weight.double() ** 2).sum()), float((m.lora_down.weight.double() ** 2).sum())) for m in sites]
    for b in batches:
        b["mask"] = b["mask"].bool()
    torch.save(dict(model_seed=0, factor_seed=6, step_seed=999, n_unet_sites=len(up) // 2, batches=batches,
                    steps=rec, factors=factors, factor_moments=sums), f"{OUT}/pti_perform_tuning.pt")
    print("tuning", [(r["loss"], r["lrs"]) for r in rec], len(sites))


def _sites(model):
    return [m for m in model.modules() if type(m).__name__.startswith("LoraInjected")]


def _load_ref(fname, modname):
    """Load one reference file as a sub-module of a stub package `lora_diffusion_ref` whose `.lora` is
    the real lora.py; `fire` and `diffusers` are empty stand-ins (only imported, never called here)."""
    stubs = {"fire": {"Fire": lambda *a, **k: None}, "diffusers": {"StableDiffusionPipeline": object}}
    planted = []
    for stub, attrs in stubs.items():
        if stub not in sys.modules:
            m = types.ModuleType(stub)
            for k, v in attrs.items():
                setattr(m, k, v)
            sys.modules[stub] = m
            planted.append(stub)
    try:
        if "lora_diffusion_ref" not in sys.modules:
            pkg = types.ModuleType("lora_diffusion_ref")
            pkg.__path__ = [f"{REF}/lora_diffusion"]
            sys.modules["lora_diffusion_ref"] = pkg
        full = f"lora_diffusion_ref.{modname}"
        if full in sys.modules:
            return sys.modules[full]
        spec = importlib.util.spec_from_file_location(full, f"{REF}/lora_diffusion/{fname}")
        mod = importlib.util.module_from_spec(spec)
        sys.modules[full] = mod
        spec.loader.exec_module(mod)
    finally:
        for stub in planted:
            sys.modules.pop(stub, None)
    return mod


def gen_live(R):
    """tests/test_vs_reference_live.py: the reference's public namespace and signatures, and its
    outputs on the tiny host models for the same seeded calls the tests make with lora_b200 (each
    side is also checked against lora_b200 here). Tensors as digests (tests/refgold.py), except the
    fp32 operator case, which is stored whole because it is compared with a tolerance."""
    import copy
    import inspect
    import tempfile
    import warnings
    from safetensors import safe_open
    import lora_b200 as L
    from lora_b200.host.clip import build_text_encoder
    from lora_b200.host.unet_sd15 import UNet2DConditionModel, UNetConfig
    from refgold import canon_metadata, canon_signature, digest
    out = {}
    tmp = tempfile.mkdtemp()

    # ---- namespace and signatures
    names = {n for n in dir(R) if not n.startswith("_") and (callable(getattr(R, n)) or n.isupper()
             or n in ("safetensors_available",))}
    skip = {"Callable", "Dict", "List", "Optional", "Set", "Tuple", "Type", "Union", "groupby", "F", "nn",
            "np", "PIL", "torch", "json", "math", "_find_modules_old"}
    out["namespace"] = sorted(n for n in names if n not in skip and not inspect.ismodule(getattr(R, n)))
    signed = ["inject_trainable_lora", "inject_trainable_lora_extended", "monkeypatch_or_replace_lora",
              "monkeypatch_or_replace_lora_extended", "patch_pipe", "save_all", "tune_lora_scale",
              "monkeypatch_add_lora", "apply_learned_embed_in_clip", "extract_lora_as_tensor",
              "LoraInjectedLinear.__init__", "LoraInjectedConv2d.__init__"]
    out["signatures"] = {}
    for n in signed:
        obj = R
        for part in n.split("."):
            obj = getattr(obj, part)
        out["signatures"][n] = canon_signature(obj)

    # ---- inject (extended unet + text encoder), save_all, load the file back, collapse
    torch.manual_seed(0)
    unet, te = UNet2DConditionModel(UNetConfig.tiny()), build_text_encoder(tiny=True)
    torch.manual_seed(1)
    _, n2 = R.inject_trainable_lora_extended(unet, r=4)
    _, t2 = R.inject_trainable_lora(te, target_replace_module={"CLIPAttention"}, r=4)
    refs = _sites(unet) + _sites(te)
    rec = {"unet_names": n2, "text_names": t2, "kinds": [type(m).__name__ for m in refs],
           "down": [digest(m.lora_down.weight) for m in refs]}
    g = torch.Generator().manual_seed(2)
    for m in refs:
        m.lora_up.weight.data.normal_(0, 0.05, generator=g)
    R.tune_lora_scale(unet, 0.7)
    path = os.path.join(tmp, "b.safetensors")
    R.save_all(unet, te, path, save_ti=False, target_replace_module_unet=R.UNET_EXTENDED_TARGET_REPLACE)
    f = safe_open(path, "pt")
    rec["saved"] = {k: digest(f.get_tensor(k)) for k in f.keys()}
    rec["saved_metadata"] = canon_metadata(f.metadata())

    class P:
        pass
    pr = P()
    torch.manual_seed(0)
    pr.unet, pr.text_encoder = UNet2DConditionModel(UNetConfig.tiny()), build_text_encoder(tiny=True)
    R.monkeypatch_or_replace_safeloras(pr, f)
    rec["loaded"] = [[type(m).__name__, digest(m.lora_up.weight), digest(m.lora_down.weight)]
                     for m in _sites(pr.unet) + _sites(pr.text_encoder)]
    R.collapse_lora(pr.unet, 0.5)
    rec["collapsed"] = [digest(m.linear.weight if hasattr(m, "linear") else m.conv.weight) for m in _sites(pr.unet)]
    out["inject_save_load"] = rec

    # ---- the reference operator classes, fp32, fwd + bwd (stored whole: compared with a tolerance)
    torch.manual_seed(3)
    ops = []
    for conv in (False, True):
        if conv:
            base = nn.Conv2d(8, 12, 3, padding=1)
            ref = R.LoraInjectedConv2d(8, 12, 3, 1, 1, r=4, dropout_p=0.0, scale=1.3)
            ref.conv.weight, ref.conv.bias = base.weight, base.bias
            x = torch.randn(2, 8, 7, 7)
        else:
            base = nn.Linear(24, 40)
            ref = R.LoraInjectedLinear(24, 40, True, r=4, dropout_p=0.0, scale=1.3)
            ref.linear.weight, ref.linear.bias = base.weight, base.bias
            x = torch.randn(3, 5, 24)
        ref.lora_up.weight.data.normal_(0, 0.1)
        x1 = x.clone().requires_grad_(True)
        y = ref(x1)
        gy = torch.randn_like(y)
        y.backward(gy)
        ops.append({k: v.detach().clone() for k, v in dict(
            W=base.weight, b=base.bias, down=ref.lora_down.weight, up=ref.lora_up.weight, x=x, gy=gy, y=y,
            dX=x1.grad, d_down=ref.lora_down.weight.grad, d_up=ref.lora_up.weight.grad).items()})
    torch.save(ops, f"{OUT}/reference_modules_fp32.pt")

    # ---- site order of the extended inject: module path and factor shapes of every site
    torch.manual_seed(0)
    u1 = UNet2DConditionModel(UNetConfig.tiny())
    R.inject_trainable_lora_extended(u1, r=4)
    out["extended_targets"] = sorted(R.UNET_EXTENDED_TARGET_REPLACE)
    out["inject_order"] = [[p, list(m.lora_up.weight.shape), list(m.lora_down.weight.shape)]
                           for p, m in u1.named_modules() if type(m).__name__.startswith("LoraInjected")]

    # ---- small helpers on the tiny UNet
    torch.manual_seed(0)
    base = UNet2DConditionModel(UNetConfig.tiny())
    ours, ref = copy.deepcopy(base), copy.deepcopy(base)
    rec = {"find_children": [[type(p).__name__, n, list(c.weight.shape)]
                             for p, n, c in R._find_children(ref, [nn.Linear, nn.Conv2d])]}
    torch.manual_seed(1)
    L.inject_trainable_lora(ours, r=4)
    torch.manual_seed(1)
    R.inject_trainable_lora(ref, r=4)
    rec["down"] = [digest(m.lora_down.weight) for m in _sites(ref)]
    g = torch.Generator().manual_seed(2)
    for so, sr in zip(_sites(ours), _sites(ref)):
        so.lora_up.weight.data.normal_(0, 0.02, generator=g)
        sr.lora_up.weight.data.copy_(so.lora_up.weight.data)
    rec["ups_down"] = [[digest(u.weight), digest(d.weight)] for u, d in R.extract_lora_ups_down(ref)]
    R.save_lora_as_json(ref, os.path.join(tmp, "r.json"))
    with open(os.path.join(tmp, "r.json"), "rb") as fh:
        rec["json_sha256"] = hashlib.sha256(fh.read()).hexdigest()
    R.save_lora_weight(ref, os.path.join(tmp, "r.pt"))
    rec["pt"] = [digest(t) for t in torch.load(os.path.join(tmp, "r.pt"))]
    emb = {"<tok>": torch.randn(48, generator=g)}
    xs = os.path.join(tmp, "x.safetensors")
    L.save_safeloras_with_embeds({"unet": (ours, L.UNET_DEFAULT_TARGET_REPLACE)}, emb, xs)
    flat = lambda d: {k: [[digest(torch.as_tensor(t)) for t in v[0]], v[1], sorted(v[2])] for k, v in d.items()}
    rec["load_safeloras"] = flat(R.load_safeloras(xs))
    rec["load_safeloras_embeds"] = {k: digest(v) for k, v in R.load_safeloras_embeds(xs).items()}
    both = R.load_safeloras_both(xs)
    rec["load_safeloras_both"] = [flat(both[0]), {k: digest(v) for k, v in both[1].items()}]
    rec["ti_lora_path"] = R._ti_lora_path("a/b.c.pt")
    rec["text_lora_path"] = R._text_lora_path("a/b.c.pt")

    class Tok:
        def __init__(self, n):
            self.v = {f"w{i}": i for i in range(n)}

        def add_tokens(self, t):
            if t in self.v:
                return 0
            self.v[t] = len(self.v)
            return 1

        def convert_tokens_to_ids(self, t):
            return self.v[t]

        def __len__(self):
            return len(self.v)
    torch.manual_seed(3)
    te_r = build_text_encoder(tiny=True)
    V = te_r.get_input_embeddings().weight.shape[0]
    torch.save(emb, os.path.join(tmp, "e.pt"))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        torch.manual_seed(4)
        R.load_learned_embed_in_clip(os.path.join(tmp, "e.pt"), te_r, Tok(V), token=None, idempotent=True)
    rec["learned_embed_table"] = digest(te_r.get_input_embeddings().weight)
    out["small_helpers"] = rec
    with open(f"{OUT}/reference_live.json", "w") as fh:
        json.dump(out, fh, indent=0)


def gen_formats(R):
    """tests/test_formats_cpu.py: lora_manager.lora_join, cli_lora_add.add and the to_ckpt_v2 key
    conversions of the reference, on the seeded LoRA files the tests write with lora_b200."""
    import tempfile
    from safetensors import safe_open
    from lora_b200.host.unet_sd15 import UNet2DConditionModel, UNetConfig
    from refgold import canon_metadata, digest
    from test_formats_cpu import _make_lora_file, _read, _vae_keys
    tmp = tempfile.mkdtemp()
    out = {}
    M = _load_ref("lora_manager.py", "lora_manager")
    p1 = _make_lora_file(os.path.join(tmp, "a.safetensors"), 3, 4, with_tokens=("<z>", "<y>"))
    p2 = _make_lora_file(os.path.join(tmp, "b.safetensors"), 4, 4)
    t, meta, ranks, toks = M.lora_join([safe_open(p, framework="pt", device="cpu") for p in (p1, p2)])
    out["join"] = {"tensors": {k: digest(v) for k, v in t.items()}, "metadata": canon_metadata(meta),
                   "ranklist": ranks, "token_sizes": toks}
    _load_ref("lora.py", "lora")
    _load_ref("to_ckpt_v2.py", "to_ckpt_v2")
    A = _load_ref("cli_lora_add.py", "cli_lora_add")
    p1 = _make_lora_file(os.path.join(tmp, "c.safetensors"), 11, 4, with_tokens=("<a>",))
    p2 = _make_lora_file(os.path.join(tmp, "d.safetensors"), 12, 4, with_tokens=("<b>",))
    out["add"] = {}
    for mode in ("lpl", "ljl"):
        r = os.path.join(tmp, f"r_{mode}.safetensors")
        A.add(p1, p2, r, 0.7, 0.4, mode=mode)
        tr, mr = _read(r)
        out["add"][mode] = {"tensors": {k: digest(v) for k, v in tr.items()}, "metadata": canon_metadata(mr)}
    C = _load_ref("to_ckpt_v2.py", "to_ckpt_v2")
    unet_sd = {k: torch.zeros(1) for k in UNet2DConditionModel(UNetConfig.tiny()).state_dict()}
    out["ckpt_unet_keys"] = list(C.convert_unet_state_dict(dict(unet_sd)))
    vae_sd = {k: (torch.zeros(4, 4) if ".attentions.0." in k and k.endswith("weight") and "group_norm" not in k
                  else torch.zeros(4)) for k in _vae_keys()}
    out["ckpt_vae"] = [[k, list(v.shape)] for k, v in C.convert_vae_state_dict(dict(vae_sd)).items()]
    with open(f"{OUT}/reference_formats.json", "w") as fh:
        json.dump(out, fh, indent=0)


GENERATORS = {"ops": gen_ops, "ctor_rng": gen_ctor_rng, "inject": gen_inject, "manifest": gen_manifest,
              "svd": gen_svd, "adamw": lambda R: gen_adamw(), "loss_step": gen_loss_step, "ti": gen_ti,
              "tuning": gen_tuning, "live": gen_live, "formats": gen_formats}

if __name__ == "__main__":
    # python scripts/make_golden.py [name ...]   (default: every generator)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    R = load_ref_lora()
    for name in sys.argv[1:] or GENERATORS:
        GENERATORS[name](R)
    for fn in sorted(os.listdir(OUT)):
        print(fn, os.path.getsize(f"{OUT}/{fn}"))
