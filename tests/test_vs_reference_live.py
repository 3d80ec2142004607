"""Side-by-side comparison with the original lora_diffusion/lora.py on the tiny host models. The
original's side of every comparison was recorded by running it on the same seeded calls
(scripts/make_golden.py -> tests/golden/reference_live.json, reference_modules_fp32.pt); tensors
are compared through content digests (tests/refgold.py), so every equality stays exact."""
import copy
import hashlib

import pytest
import torch
import torch.nn as nn
from safetensors import safe_open

import lora_b200 as L
from lora_b200.host.clip import build_text_encoder
from lora_b200.host.unet_sd15 import UNet2DConditionModel, UNetConfig
from oracle.ref_modules import RefLoraSite, ref_inject
from refgold import GOLD, canon_metadata, canon_signature, digest, load


@pytest.fixture(scope="module")
def G():
    return load("reference_live.json")


def _sites(model):
    return [m for m in model.modules() if type(m).__name__.startswith("LoraInjected")]


def test_public_names_cover_the_reference_namespace(G):
    missing = sorted(n for n in G["namespace"] if not hasattr(L, n))
    assert missing == [], missing
    for name, want in G["signatures"].items():
        obj = L
        for part in name.split("."):
            obj = getattr(obj, part)
        assert canon_signature(obj) == want, name      # names, order and defaults


def test_inject_save_load_equal_reference_on_tiny_models(G, tmp_path):
    g0 = G["inject_save_load"]
    torch.manual_seed(0)
    unet = UNet2DConditionModel(UNetConfig.tiny())
    te = build_text_encoder(tiny=True)
    torch.manual_seed(1)
    _, n1 = L.inject_trainable_lora_extended(unet, r=4)
    _, t1 = L.inject_trainable_lora(te, target_replace_module={"CLIPAttention"}, r=4)
    assert n1 == g0["unet_names"] and t1 == g0["text_names"]
    ours = _sites(unet) + _sites(te)
    assert [type(m).__name__ for m in ours] == g0["kinds"]
    # same RNG consumption => identical initial factors
    assert [digest(m.lora_down.weight) for m in ours] == g0["down"]
    g = torch.Generator().manual_seed(2)
    for a in ours:
        a.lora_up.weight.data.normal_(0, 0.05, generator=g)
    L.tune_lora_scale(unet, 0.7)
    L.save_all(unet, te, str(tmp_path / "a.safetensors"), save_ti=False,
               target_replace_module_unet=L.UNET_EXTENDED_TARGET_REPLACE)
    fa = safe_open(str(tmp_path / "a.safetensors"), "pt")
    assert sorted(fa.keys()) == sorted(g0["saved"])
    assert {k: digest(fa.get_tensor(k)) for k in fa.keys()} == g0["saved"]
    # same keys, tensors and metadata as the reference's file: the reference's loader would read ours
    # exactly as it read its own, which is what "loaded" recorded
    assert canon_metadata(fa.metadata()) == g0["saved_metadata"]

    class P:
        pass
    po = P()
    torch.manual_seed(0)
    po.unet, po.text_encoder = UNet2DConditionModel(UNetConfig.tiny()), build_text_encoder(tiny=True)
    L.monkeypatch_or_replace_safeloras(po, fa)
    got = [[type(m).__name__, digest(m.lora_up.weight), digest(m.lora_down.weight)]
           for m in _sites(po.unet) + _sites(po.text_encoder)]
    assert got == g0["loaded"]
    L.collapse_lora(po.unet, 0.5)
    assert [digest(m.linear.weight if hasattr(m, "linear") else m.conv.weight)
            for m in _sites(po.unet)] == g0["collapsed"]


def test_oracle_modules_equal_reference_modules_fp32():
    """oracle/ref_modules.RefLoraSite vs the reference operator classes, random inputs, fwd+bwd."""
    cases = torch.load(f"{GOLD}/reference_modules_fp32.pt")
    assert len(cases) == 2
    for c in cases:
        if c["W"].dim() == 4:
            base = nn.Conv2d(8, 12, 3, padding=1)
        else:
            base = nn.Linear(24, 40)
        base.weight.data.copy_(c["W"]); base.bias.data.copy_(c["b"])
        site = RefLoraSite(base, r=4, dropout_p=0.0, scale=1.3)
        site.down.data.copy_(c["down"]); site.up.data.copy_(c["up"])
        x = c["x"].clone().requires_grad_(True)
        y = site(x)
        y.backward(c["gy"])
        assert torch.allclose(c["y"], y, atol=1e-5)
        assert torch.allclose(c["dX"], x.grad, atol=1e-5)
        assert torch.allclose(c["d_down"], site.down.grad, atol=1e-5)
        assert torch.allclose(c["d_up"], site.up.grad, atol=1e-5)


def test_oracle_inject_order_equals_reference(G):
    torch.manual_seed(0)
    u2 = UNet2DConditionModel(UNetConfig.tiny())
    plain = copy.deepcopy(u2)
    sites = ref_inject(u2, set(G["extended_targets"]), r=4, extended=True)
    assert len(sites) == len(G["inject_order"])
    for a, (path, up, down) in zip(sites, G["inject_order"]):
        assert list(a.up.shape) == up and list(a.down.shape) == down
        # the reference's site at `path` wraps the layer found there in the un-injected model
        assert a.weight is not None and torch.equal(a.weight, plain.get_submodule(path).weight)


def test_small_helpers_equal_reference(G, tmp_path):
    """The remaining small public functions, side by side with the reference on the tiny UNet:
    _find_children, extract_lora_ups_down, save_lora_as_json, save_lora_weight (.pt),
    load_safeloras / load_safeloras_embeds / load_safeloras_both, _ti_lora_path,
    load_learned_embed_in_clip."""
    g0 = G["small_helpers"]
    torch.manual_seed(0)
    ours = UNet2DConditionModel(UNetConfig.tiny())
    # _find_children: same (parent, name, child) walk on an un-injected model
    a = [[type(p).__name__, n, list(c.weight.shape)] for p, n, c in L._find_children(ours, [nn.Linear, nn.Conv2d])]
    assert a == g0["find_children"] and len(a) > 20
    torch.manual_seed(1)
    L.inject_trainable_lora(ours, r=4)
    assert [digest(s.lora_down.weight) for s in _sites(ours)] == g0["down"]      # ctor RNG parity
    g = torch.Generator().manual_seed(2)
    for so in _sites(ours):
        so.lora_up.weight.data.normal_(0, 0.02, generator=g)
    eo = L.extract_lora_ups_down(ours)
    assert len(eo) == len(_sites(ours))
    assert [[digest(u.weight), digest(d.weight)] for u, d in eo] == g0["ups_down"]
    # json / .pt writers: identical bytes (json) and identical tensors (.pt)
    L.save_lora_as_json(ours, str(tmp_path / "o.json"))
    assert hashlib.sha256((tmp_path / "o.json").read_bytes()).hexdigest() == g0["json_sha256"]
    L.save_lora_weight(ours, str(tmp_path / "o.pt"))
    assert [digest(t) for t in torch.load(tmp_path / "o.pt")] == g0["pt"]
    # safetensors loaders
    emb = {"<tok>": torch.randn(48, generator=g)}
    L.save_safeloras_with_embeds({"unet": (ours, L.UNET_DEFAULT_TARGET_REPLACE)}, emb, str(tmp_path / "x.safetensors"))
    flat = lambda d: {k: [[digest(torch.as_tensor(t)) for t in v[0]], v[1], sorted(v[2])] for k, v in d.items()}
    xs = str(tmp_path / "x.safetensors")
    assert flat(L.load_safeloras(xs)) == g0["load_safeloras"]
    assert {k: digest(v) for k, v in L.load_safeloras_embeds(xs).items()} == g0["load_safeloras_embeds"]
    both = L.load_safeloras_both(xs)
    assert [flat(both[0]), {k: digest(v) for k, v in both[1].items()}] == g0["load_safeloras_both"]
    assert L._ti_lora_path("a/b.c.pt") == g0["ti_lora_path"]
    assert L._text_lora_path("a/b.c.pt") == g0["text_lora_path"]
    # learned-embedding loader on a tiny text encoder with a duck tokenizer
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
    te_o = build_text_encoder(tiny=True)
    V = te_o.get_input_embeddings().weight.shape[0]
    torch.save(emb, tmp_path / "e.pt")
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        torch.manual_seed(4)
        L.load_learned_embed_in_clip(str(tmp_path / "e.pt"), te_o, Tok(V), token=None, idempotent=True)
    assert digest(te_o.get_input_embeddings().weight) == g0["learned_embed_table"]
    assert torch.equal(te_o.get_input_embeddings().weight[V], emb["<tok>"])
