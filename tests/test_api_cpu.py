"""Host-side API of lora_b200 against artefacts produced by the real reference
(tests/golden, scripts/make_golden.py). CPU only: no forward pass is executed here
(lora_b200 has no CPU compute path)."""
import json
import os

import pytest
import torch
import torch.nn as nn
from safetensors import safe_open

import lora_b200 as L
from lora_b200.host.clip import build_text_encoder
from lora_b200.host.unet_sd15 import UNet2DConditionModel, UNetConfig

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _sites(model):
    return [m for m in model.modules() if type(m).__name__.startswith("LoraInjected")]


def test_constructor_consumes_rng_like_the_reference():
    """Seed parity (SURVEY.md 7): after manual_seed(0) the down factor and the NEXT random draw
    equal the reference's (it burns three kaiming inits before normal_, lora.py:43-50)."""
    g = torch.load(f"{GOLD}/ctor_rng.pt")
    torch.manual_seed(0)
    m = L.LoraInjectedLinear(16, 24, True, r=4)
    assert torch.equal(m.lora_down.weight.detach(), g["linear_down"])
    assert torch.equal(torch.rand(3), g["linear_next_rand"])
    assert torch.count_nonzero(m.lora_up.weight) == 0
    torch.manual_seed(0)
    c = L.LoraInjectedConv2d(8, 12, 3, 1, 1, r=4)
    assert torch.equal(c.lora_down.weight.detach(), g["conv_down"])
    assert torch.equal(torch.rand(3), g["conv_next_rand"])
    assert c.lora_down.weight.shape == (4, 8, 3, 3) and c.lora_up.weight.shape == (12, 4, 1, 1)


def test_constructor_contract():
    with pytest.raises(ValueError):
        L.LoraInjectedLinear(8, 4, r=5)
    with pytest.raises(ValueError):
        L.LoraInjectedConv2d(4, 16, 3, r=8)
    m = L.LoraInjectedLinear(8, 8, bias=True, r=2)
    assert set(dict(m.named_children())) == {"linear", "lora_down", "dropout", "lora_up", "selector"}
    assert set(m.state_dict()) == {"linear.weight", "linear.bias", "lora_down.weight", "lora_up.weight"}
    assert m.dropout.p == 0.1 and m.scale == 1.0 and m.training
    c = L.LoraInjectedConv2d(8, 8, 3, r=2)
    assert set(dict(c.named_children())) == {"conv", "lora_down", "dropout", "lora_up", "selector"}
    up, down = m.realize_as_lora()
    assert up.shape == (8, 2) and down.shape == (2, 8)
    m.set_selector_from_diag(torch.tensor([2.0, 3.0]))
    assert torch.equal(m.selector.weight.data, torch.diag(torch.tensor([2.0, 3.0])))
    with pytest.raises(AssertionError):
        m.set_selector_from_diag(torch.ones(3))


def test_inject_order_matches_reference_golden():
    g = json.load(open(f"{GOLD}/inject_tiny.json"))
    torch.manual_seed(0)
    unet = UNet2DConditionModel(UNetConfig.tiny())
    frozen_before = {id(p) for p in unet.parameters()}
    params, names = L.inject_trainable_lora(unet, r=4)
    assert names == g["unet_default_names"]
    shapes = [[list(m.lora_up.weight.shape), list(m.lora_down.weight.shape)] for m in _sites(unet)]
    assert shapes == g["unet_default_shapes"]
    assert len(params) == 2 * len(names)
    flat = [p for gen in params for p in gen]
    assert all(p.requires_grad for p in flat)
    # frozen Parameters are shared, not copied (lora.py:290-292)
    assert all(id(m.linear.weight) in frozen_before for m in _sites(unet))
    # default dropout of inject_trainable_lora is 0.0 (lora.py:261)
    assert all(m.dropout.p == 0.0 for m in _sites(unet))

    torch.manual_seed(0)
    unet2 = UNet2DConditionModel(UNetConfig.tiny())
    _, names2 = L.inject_trainable_lora_extended(unet2, r=4)
    assert names2 == g["unet_extended_names"]
    assert [type(m).__name__ for m in _sites(unet2)] == g["unet_extended_kinds"]
    assert [[list(m.lora_up.weight.shape), list(m.lora_down.weight.shape)] for m in _sites(unet2)] == g["unet_extended_shapes"]
    assert all(m.dropout.p == 0.1 for m in _sites(unet2))      # class default (lora.py:334-356)

    torch.manual_seed(0)
    te = build_text_encoder(tiny=True)
    _, names3 = L.inject_trainable_lora(te, target_replace_module={"CLIPAttention"}, r=4)
    assert names3 == g["text_names"]


def _rebuild_tiny_state():
    raw = torch.load(f"{GOLD}/tiny_saved_raw.pt")
    torch.manual_seed(0)
    unet = UNet2DConditionModel(UNetConfig.tiny())
    te = build_text_encoder(tiny=True)
    L.inject_trainable_lora(unet, r=4)
    L.inject_trainable_lora(te, target_replace_module={"CLIPAttention"}, r=4)
    for key, mdl in (("unet", unet), ("text_encoder", te)):
        for m, (up, down) in zip(_sites(mdl), raw[key]):
            m.lora_up.weight.data.copy_(up)
            m.lora_down.weight.data.copy_(down)
    L.tune_lora_scale(unet, 0.5)
    return unet, te


def test_saved_safetensors_equal_the_reference_file(tmp_path):
    """Same state saved by our save_safeloras_with_embeds vs the reference's file: identical key
    set, identical tensor bytes (fp16, up pre-multiplied by scale), identical metadata (target
    lists compared as sets: the reference dumps list(set))."""
    unet, te = _rebuild_tiny_state()
    out = str(tmp_path / "ours.safetensors")
    L.save_safeloras_with_embeds({"unet": (unet, L.DEFAULT_TARGET_REPLACE),
                                  "text_encoder": (te, L.TEXT_ENCODER_DEFAULT_TARGET_REPLACE)},
                                 {"<s1>": torch.arange(48, dtype=torch.float32)}, out)
    a = safe_open(out, framework="pt")
    b = safe_open(f"{GOLD}/tiny_saved.safetensors", framework="pt")
    assert sorted(a.keys()) == sorted(b.keys())
    for k in a.keys():
        ta, tb = a.get_tensor(k), b.get_tensor(k)
        assert ta.dtype == tb.dtype and torch.equal(ta, tb), k
    ma, mb = a.metadata(), b.metadata()
    assert set(ma) == set(mb)
    for k in ma:
        if k in ("unet", "text_encoder"):
            assert set(json.loads(ma[k])) == set(json.loads(mb[k]))
        else:
            assert ma[k] == mb[k]


def test_parse_and_monkeypatch_roundtrip(tmp_path):
    """parse_safeloras on the reference-written file, monkeypatch into a fresh model, re-save:
    the factors survive; ranks/targets parsed; embeds parsed."""
    f = safe_open(f"{GOLD}/tiny_saved.safetensors", framework="pt")
    parsed = L.parse_safeloras(f)
    assert set(parsed) == {"unet", "text_encoder"}
    w, ranks, targets = parsed["unet"]
    assert len(w) == 2 * len(ranks) and set(ranks) == {4}
    assert set(targets) == set(L.DEFAULT_TARGET_REPLACE)
    emb = L.parse_safeloras_embeds(f)
    assert list(emb) == ["<s1>"] and torch.equal(emb["<s1>"], torch.arange(48, dtype=torch.float32))

    class Pipe:
        pass
    torch.manual_seed(0)
    pipe = Pipe()
    pipe.unet = UNet2DConditionModel(UNetConfig.tiny())
    pipe.text_encoder = build_text_encoder(tiny=True)
    L.monkeypatch_or_replace_safeloras(pipe, f)
    sites = _sites(pipe.unet)
    assert len(sites) == len(ranks)
    assert all(s.dropout.p == 0.1 and s.scale == 1.0 and s.training for s in sites)  # lora.py:689-694
    for i, s in enumerate(sites):
        assert torch.equal(s.lora_up.weight.data.half(), f.get_tensor(f"unet:{i}:up"))
        assert torch.equal(s.lora_down.weight.data.half(), f.get_tensor(f"unet:{i}:down"))
    # replace again (sites are already LoRA modules) -> still the same number of sites
    L.monkeypatch_or_replace_safeloras(pipe, f)
    assert len(_sites(pipe.unet)) == len(ranks)
    # remove -> plain layers sharing the frozen weights
    w0 = sites[0].linear.weight
    L.monkeypatch_remove_lora(pipe.unet)
    assert len(_sites(pipe.unet)) == 0
    assert any(p is w0 for p in pipe.unet.parameters())


def test_pt_format_and_resume(tmp_path):
    unet, te = _rebuild_tiny_state()
    path = str(tmp_path / "lora.pt")
    L.save_lora_weight(unet, path)
    flat = torch.load(path)
    sites = _sites(unet)
    assert len(flat) == 2 * len(sites) and all(t.dtype == torch.float16 for t in flat)
    assert torch.equal(flat[0], sites[0].lora_up.weight.data.half())        # raw, NOT scaled
    assert torch.equal(flat[1], sites[0].lora_down.weight.data.half())
    torch.manual_seed(0)
    fresh = UNet2DConditionModel(UNetConfig.tiny())
    L.inject_trainable_lora(fresh, r=4, loras=path)
    f_sites = _sites(fresh)
    assert torch.equal(f_sites[3].lora_up.weight.data, flat[6]) and f_sites[3].lora_up.weight.requires_grad
    # .pt -> safetensors converter
    out = str(tmp_path / "conv.safetensors")
    L.convert_loras_to_safeloras({"unet": (path, L.DEFAULT_TARGET_REPLACE, 4)}, out)
    g = safe_open(out, framework="pt")
    assert g.metadata()["unet:0:rank"] == "4" and torch.equal(g.get_tensor("unet:2:down"), flat[5])
    # save_all in both forms
    L.save_all(unet, te, str(tmp_path / "all.safetensors"), save_ti=False)
    h = safe_open(str(tmp_path / "all.safetensors"), framework="pt")
    assert f"text_encoder:{len(_sites(te)) - 1}:up" in h.keys()
    L.save_all(unet, te, str(tmp_path / "all.pt"), save_ti=False, safe_form=False)
    assert os.path.exists(str(tmp_path / "all.text_encoder.pt"))


def test_collapse_add_scale_diag_inspect():
    from oracle import lora_ops as O
    torch.manual_seed(1)

    class Attention(nn.Module):
        def __init__(self):
            super().__init__()
            self.to_q = nn.Linear(16, 16, bias=False)

    class ResnetBlock2D(nn.Module):
        def __init__(self):
            super().__init__()
            self.conv1 = nn.Conv2d(8, 8, 3, padding=1)

    model = nn.Sequential(Attention(), ResnetBlock2D())
    L.inject_trainable_lora_extended(model, r=4)
    lin, conv = _sites(model)
    lin.lora_up.weight.data.normal_(); conv.lora_up.weight.data.normal_()
    w_lin, w_conv = lin.linear.weight.data.clone(), conv.conv.weight.data.clone()
    L.collapse_lora(model, alpha=0.5)
    d_lin = O.collapse_delta(lin.lora_down.weight, lin.lora_up.weight, 0.5)
    d_conv = O.collapse_delta(conv.lora_down.weight, conv.lora_up.weight, 0.5)
    assert torch.allclose(lin.linear.weight.data.double(), w_lin.double() + d_lin, atol=1e-5)
    assert torch.allclose(conv.conv.weight.data.double(), w_conv.double() + d_conv.reshape(w_conv.shape), atol=1e-5)
    L.tune_lora_scale(model, 0.25)
    assert lin.scale == 0.25 and conv.scale == 0.25
    L.set_lora_diag(model, torch.tensor([1.0, 2.0, 3.0, 4.0]))
    assert isinstance(lin.selector, nn.Linear) and isinstance(conv.selector, nn.Conv2d)
    moved = L.inspect_lora(model)
    assert len(moved) == 2 and all(v[0] > 0 for v in moved.values())
    up0, down0 = lin.lora_up.weight.data.clone(), lin.lora_down.weight.data.clone()
    L.monkeypatch_add_lora(model, [torch.ones(16, 4), torch.ones(4, 16)], {"Attention"}, alpha=2.0, beta=0.5)
    assert torch.allclose(lin.lora_up.weight.data, 2.0 * torch.ones(16, 4) + 0.5 * up0)
    assert torch.allclose(lin.lora_down.weight.data, 2.0 * torch.ones(4, 16) + 0.5 * down0)


def test_fixture_manifest_layout(tmp_path):
    """The ten fixture files of the reference pin the on-disk layout (SURVEY.md 4). The manifest
    (keys, shapes, dtypes, metadata, what the reference's own parse_safeloras returned) travels
    with the repo; our parser runs on a file of each manifest's layout (its keys, shapes, dtypes and
    metadata; zero tensors, the parser reads no values)."""
    from safetensors.torch import save_file
    man = json.load(open(f"{GOLD}/example_loras_manifest.json"))
    assert len(man) == 10
    torch.manual_seed(0)
    with torch.device("meta"):
        unet = UNet2DConditionModel(UNetConfig.sd15())
    L.inject_trainable_lora(unet, r=4)
    sites = _sites(unet)
    for fn, ent in man.items():
        keys = ent["tensors"]
        n_unet = len([k for k in keys if k.startswith("unet:")]) // 2
        assert n_unet == 144 == len(sites)
        assert len([k for k in keys if k.startswith("text_encoder:")]) == 96
        for i, s in enumerate(sites):     # our host UNet reproduces the site order of every file
            r = int(ent["metadata"][f"unet:{i}:rank"])
            assert keys[f"unet:{i}:up"][0] == [s.linear.out_features, r]
            assert keys[f"unet:{i}:down"][0] == [r, s.linear.in_features]
        assert set(json.loads(ent["metadata"]["unet"])) == set(L.UNET_DEFAULT_TARGET_REPLACE)
        assert json.loads(ent["metadata"]["text_encoder"]) == ["CLIPAttention"]
        path = str(tmp_path / fn)
        save_file({k: torch.zeros(shape, dtype=getattr(torch, dt)) for k, (shape, dt, _) in keys.items()},
                  path, metadata=ent["metadata"])
        f = safe_open(path, framework="pt")
        ours = L.parse_safeloras(f)
        assert sorted(ours) == sorted(ent["parsed"])
        for name, info in ent["parsed"].items():
            w, ranks, targets = ours[name]
            assert len(w) == info["n_weights"] and ranks == info["ranks"] and sorted(targets) == info["targets"]
        assert sorted(L.parse_safeloras_embeds(f)) == ent["embeds"]


def test_lr_schedule_restates_diffusers_linear_and_constant():
    """cli_lora_pti.py:730-741 uses get_scheduler('linear'/'constant'); the multipliers are restated."""
    from lora_b200.train import LoraTrainStep, StepConfig

    class Dummy:
        lr_multiplier = LoraTrainStep.lr_multiplier
    d = Dummy()
    d.cfg = StepConfig(lr_scheduler="linear", lr_warmup_steps=10, max_train_steps=110)
    assert d.lr_multiplier(0) == 0.0 and d.lr_multiplier(5) == 0.5 and d.lr_multiplier(10) == 1.0
    assert abs(d.lr_multiplier(60) - 0.5) < 1e-12 and d.lr_multiplier(110) == 0.0 and d.lr_multiplier(500) == 0.0
    d.cfg = StepConfig(lr_scheduler="constant")
    assert d.lr_multiplier(0) == 1.0 and d.lr_multiplier(10 ** 6) == 1.0
    # diffusers' "constant" ignores num_warmup_steps: the reference's defaults (constant, 500 warm-up
    # steps; train_lora_dreambooth.py:345-356) mean NO warm-up
    d.cfg = StepConfig(lr_scheduler="constant", lr_warmup_steps=500)
    assert d.lr_multiplier(0) == 1.0 and d.lr_multiplier(3) == 1.0
    d.cfg = StepConfig(lr_scheduler="constant_with_warmup", lr_warmup_steps=4)
    assert [d.lr_multiplier(k) for k in (0, 1, 2, 4, 9)] == [0.0, 0.25, 0.5, 1.0, 1.0]
    d.cfg = StepConfig(lr_scheduler="cosine")
    import pytest
    with pytest.raises(ValueError):
        d.lr_multiplier(1)


def test_injected_model_survives_deepcopy_and_pickle(tmp_path):
    """Runtime caches / parent back-references must not break copy.deepcopy or torch.save of a model."""
    import copy
    import io
    torch.manual_seed(0)
    unet = UNet2DConditionModel(UNetConfig.tiny())
    L.inject_trainable_lora_extended(unet, r=4)
    twin = copy.deepcopy(unet)
    a, b = _sites(unet), _sites(twin)
    assert len(a) == len(b) and all(x is not y for x, y in zip(a, b))
    assert all(torch.equal(x.lora_down.weight, y.lora_down.weight) for x, y in zip(a, b))
    assert all(y._lb.parent is None and not y._lb.w for y in b)        # fresh runtime state
    assert L.link_sites(twin) == len(b)
    holders = {id(m) for m in twin.modules()}
    assert all(id(y._lb.parent()) in holders and y in y._lb.parent()._modules.values() for y in b)
    buf = io.BytesIO()
    torch.save(unet, buf)
    buf.seek(0)
    back = torch.load(buf, weights_only=False)
    assert [type(m).__name__ for m in _sites(back)] == [type(m).__name__ for m in a]


@pytest.mark.parametrize("inpaint,masked,prior", [(False, False, False), (False, True, False), (True, False, False),
                                                  (True, True, False), (False, False, True)])
def test_train_step_forward_backward_body_on_cpu_doubles(inpaint, masked, prior):
    """lora_b200.train.LoraTrainStep._fwd_bwd (noise draw, t_multiplier, inpainting concat, masked
    loss, set_loss_mask's resize) exercised WITHOUT a GPU: the object is assembled by hand around
    CPU host models whose LoRA sites are the oracle's eager modules (the product's own modules have
    no CPU path), and its loss is compared with oracle/ref_step.py -- itself pinned to the
    reference's `loss_step` -- for the same seed. Covers the Python of the step engine that the
    GPU-only tests would otherwise be the first to execute."""
    from lora_b200.host.clip import build_text_encoder
    from lora_b200.host.ddpm import DDPMNoiser
    from lora_b200.train import LoraTrainStep, StepConfig
    from oracle.ref_modules import ref_inject
    from oracle.ref_step import RefDreamboothStep
    torch.manual_seed(0)
    cfg_u = UNetConfig.tiny()
    cfg_u.in_channels = 9 if inpaint else 4
    unet, text = UNet2DConditionModel(cfg_u), build_text_encoder(tiny=True)
    us = ref_inject(unet, {"CrossAttention", "Attention", "GEGLU"}, r=4)
    ts = ref_inject(text, {"CLIPAttention"}, r=4)
    g = torch.Generator().manual_seed(1)
    for s in us + ts:
        s.up.data.normal_(0, 0.05, generator=g)
    shape = (2, 4, 8, 8)
    tr = object.__new__(LoraTrainStep)              # no arena / CUDA buffers: only what _fwd_bwd touches
    tr.cfg = StepConfig(use_cuda_graph=False, t_multiplier=0.8, use_mask=masked, mask_temperature=2.0,
                        train_inpainting=inpaint, with_prior_preservation=prior, prior_loss_weight=0.7)
    tr.unet, tr.text_encoder, tr.device = unet, text, torch.device("cpu")
    tr.noiser, tr.model_dtype, tr._side = DDPMNoiser(device="cpu"), torch.float32, None
    tr.latents = torch.randn(shape, generator=g) * 0.18215
    tr.input_ids = torch.randint(0, 1000, (2, 77), generator=g)
    tr.loss = torch.zeros(())
    tr.mask = torch.ones(2, 1, 8, 8)
    kw = {}
    if masked:
        img_mask = (torch.rand(2, 1, 64, 64, generator=g) > 0.4).float()
        tr.set_loss_mask(img_mask)
        kw.update(loss_mask=img_mask, mask_temperature=2.0)
    if inpaint:
        tr.inpaint_mask = (torch.rand(2, 1, 8, 8, generator=g) > 0.5).float()
        tr.masked_latents = torch.randn(shape, generator=g) * 0.18215
        kw.update(inpaint=(tr.inpaint_mask, tr.masked_latents))
    if prior:
        kw.update(prior_loss_weight=0.7)
    ref = RefDreamboothStep(unet, text, DDPMNoiser(device="cpu"), us, ts, t_multiplier=0.8)
    torch.manual_seed(77)
    noise = torch.randn(shape)
    t = torch.randint(0, 800, (2,)).long()
    want = ref.forward_loss(tr.latents, tr.input_ids, noise, t, **kw)
    want.backward()
    g_ref = torch.cat([p.grad.flatten() for p in ref.unet_params + ref.text_params])
    ref.opt.zero_grad()
    torch.manual_seed(77)
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")             # torch.autocast("cuda", enabled=False) on a CPU-only box
        tr._fwd_bwd()
    g_ours = torch.cat([p.grad.flatten() for p in ref.unet_params + ref.text_params])
    assert abs(float(tr.loss) - float(want)) <= 1e-5 * abs(float(want))
    # channels_last input on our side: a different (equally valid) fp32 convolution order
    assert float((g_ours - g_ref).norm() / g_ref.norm()) < 1e-4


def test_lr_step_first_selects_the_pti_schedule_order():
    """cli_lora_pti.perform_tuning steps the scheduler BEFORE the update (iteration k runs at
    lambda(k+1)); train_lora_dreambooth.py steps it after (lambda(k)). The golden of the real
    perform_tuning loop recorded lrs 1e-4 * (1 - k/6) for k = 1, 2, 3."""
    import os
    from lora_b200.train import LoraTrainStep, StepConfig
    G = torch.load(os.path.join(os.path.dirname(__file__), "golden", "pti_perform_tuning.pt"))

    class Arena:
        base_lr = [1e-4, 1e-5]

        def set_lr(self, lrs):
            self.seen.append(list(lrs))

    for first, offset in ((True, 1), (False, 0)):
        tr = object.__new__(LoraTrainStep)
        tr.cfg = StepConfig(lr_scheduler="linear", lr_warmup_steps=0, max_train_steps=6, lr_step_first=first)
        tr.arena, tr.global_step, tr.graph = Arena(), 0, None
        tr.arena.seen = []
        tr.loss = None
        tr._body = lambda: None
        for _ in range(3):
            tr.step_device()
        want = [[1e-4 * (1 - (k + offset) / 6), 1e-5 * (1 - (k + offset) / 6)] for k in range(3)]
        assert all(abs(a - b) < 1e-18 for got, w in zip(tr.arena.seen, want) for a, b in zip(got, w))
        if first:       # exactly what the reference loop used
            assert all(abs(a - b) < 1e-12 for got, st in zip(tr.arena.seen, G["steps"]) for a, b in zip(got, st["lrs"]))


def test_latent_cache_restates_cached_latents_branch():
    """cli_lora_pti.py:141-151: latents = vae.encode(image).latent_dist.sample() * 0.18215, once per item."""
    from lora_b200.step_ops import LatentCache

    class _Dist:
        def __init__(self, x):
            self.x = x

        def sample(self):
            return self.x[:, :4, ::8, ::8] * 2.0

    class _Enc:
        def __init__(self, x):
            self.latent_dist = _Dist(x)

    class _VAE(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.w = torch.nn.Parameter(torch.zeros(1))
            self.calls = 0

        def encode(self, x):
            self.calls += 1
            return _Enc(x)

    vae = _VAE()
    data = [{"instance_images": torch.randn(4, 64, 64), "instance_prompt_ids": torch.tensor([1, 2, 3])} for _ in range(3)]
    cache = LatentCache().build(vae, data)
    assert len(cache) == 3 and vae.calls == 3
    for item, src in zip(cache.items, data):
        assert item["instance_images"].shape == (4, 8, 8)
        assert torch.allclose(item["instance_images"], src["instance_images"][:4, ::8, ::8] * 2.0 * 0.18215)
        assert torch.equal(item["instance_prompt_ids"], src["instance_prompt_ids"])
    assert data[0]["instance_images"].shape == (4, 64, 64)          # the dataset itself is not modified
