"""SURVEY.md 8(f) ranks 2 and 4, host side: LoRA file arithmetic (`lora_add` lpl / ljl), rank-join
(`lora_manager.lora_join`, `LoRAManager`), `.pt` -> safetensors, diffusers -> CompVis `.ckpt` key
conversion. The committed example-shaped fixtures and algebraic properties are checked, and the
results of the original modules on the same seeded files, recorded by scripts/make_golden.py in
tests/golden/reference_formats.json, are compared exactly (tensors through digests, tests/refgold.py)."""
import os
import types

import pytest
import torch
from safetensors import safe_open
from safetensors.torch import save_file

import lora_b200 as L
from lora_b200 import lora_add, lora_manager, pt_to_safetensors, to_ckpt
from lora_b200.host.clip import build_text_encoder
from lora_b200.host.unet_sd15 import UNet2DConditionModel, UNetConfig
from refgold import canon_metadata, digest, load


@pytest.fixture(scope="module")
def G():
    return load("reference_formats.json")


def _make_lora_file(path, seed, r, with_tokens=()):
    torch.manual_seed(seed)
    unet = UNet2DConditionModel(UNetConfig.tiny())
    te = build_text_encoder(tiny=True)
    L.inject_trainable_lora(unet, r=r)
    L.inject_trainable_lora(te, r=r, target_replace_module=L.TEXT_ENCODER_DEFAULT_TARGET_REPLACE)
    g = torch.Generator().manual_seed(seed + 100)
    for m in list(unet.modules()) + list(te.modules()):
        if type(m).__name__ == "LoraInjectedLinear":
            m.lora_up.weight.data = torch.randn(m.lora_up.weight.shape, generator=g) * 0.05
    embeds = {t: torch.randn(te.get_input_embeddings().weight.shape[1], generator=g) for t in with_tokens}
    L.save_safeloras_with_embeds({"unet": (unet, L.UNET_DEFAULT_TARGET_REPLACE),
                                  "text_encoder": (te, L.TEXT_ENCODER_DEFAULT_TARGET_REPLACE)},
                                 embeds, path)
    return path


def _read(path):
    f = safe_open(path, framework="pt", device="cpu")
    return {k: f.get_tensor(k) for k in f.keys()}, dict(f.metadata())


# ------------------------------------------------------------------------------------- lora_join
def test_join_is_sum_of_branches_and_relabels_tokens(tmp_path):
    p1 = _make_lora_file(str(tmp_path / "a.safetensors"), 1, 4, with_tokens=("<krk>", "<a2>"))
    p2 = _make_lora_file(str(tmp_path / "b.safetensors"), 2, 2, with_tokens=("<s>",))
    f1, f2 = (safe_open(p, framework="pt", device="cpu") for p in (p1, p2))
    tensors, meta, ranklist, toks = lora_manager.lora_join([f1, f2])
    assert ranklist == [4, 2] and toks == [2, 1]
    t1, _ = _read(p1)
    t2, _ = _read(p2)
    n_sites = 0
    for k in t1:
        if not k.endswith(":up"):
            continue
        n_sites += 1
        d = k[:-2] + "down"
        joined = tensors[k].float() @ tensors[d].float()
        want = t1[k].float() @ t1[d].float() + t2[k].float() @ t2[d].float()
        assert torch.allclose(joined, want, atol=1e-5)
        assert meta[k[:-2] + "rank"] == "6"
    assert n_sites > 10
    # tokens: sorted within a file, renamed <s{file}-{j}>, originals gone
    assert torch.equal(tensors["<s0-0>"], t1["<a2>"]) and torch.equal(tensors["<s0-1>"], t1["<krk>"])
    assert torch.equal(tensors["<s1-0>"], t2["<s>"])
    assert meta["<s0-0>"] == meta["<s1-0>"] == "<embed>" and "<krk>" not in meta and "<krk>" not in tensors


def test_join_rejects_mixed_ranks_inside_one_file():
    bad = lora_manager.DummySafeTensorObject({}, {"unet:0:rank": "4", "unet:1:rank": "8"})
    with pytest.raises(AssertionError):
        lora_manager.lora_join([bad])


def test_join_equals_reference(G, tmp_path):
    ref = G["join"]
    p1 = _make_lora_file(str(tmp_path / "a.safetensors"), 3, 4, with_tokens=("<z>", "<y>"))
    p2 = _make_lora_file(str(tmp_path / "b.safetensors"), 4, 4)
    ours = lora_manager.lora_join([safe_open(p, framework="pt", device="cpu") for p in (p1, p2)])
    assert canon_metadata(ours[1]) == ref["metadata"] and ours[2] == ref["ranklist"] and ours[3] == ref["token_sizes"]
    assert ours[0].keys() == ref["tensors"].keys()
    assert {k: digest(v) for k, v in ours[0].items()} == ref["tensors"]


class _Tok:
    """Minimal tokenizer double with the three calls apply_learned_embed_in_clip makes."""
    def __init__(self, n):
        self.vocab = {f"w{i}": i for i in range(n)}

    def add_tokens(self, t):
        if t in self.vocab:
            return 0
        self.vocab[t] = len(self.vocab)
        return 1

    def convert_tokens_to_ids(self, t):
        return self.vocab[t]

    def __len__(self):
        return len(self.vocab)


def test_manager_patches_joined_lora_and_tunes_per_file_strength(tmp_path):
    p1 = _make_lora_file(str(tmp_path / "a.safetensors"), 5, 4, with_tokens=("<a>",))
    p2 = _make_lora_file(str(tmp_path / "b.safetensors"), 6, 2, with_tokens=("<b>", "<c>"))
    torch.manual_seed(0)
    te = build_text_encoder(tiny=True)
    pipe = types.SimpleNamespace(unet=UNet2DConditionModel(UNetConfig.tiny()), text_encoder=te,
                                 tokenizer=_Tok(te.get_input_embeddings().weight.shape[0]))
    mgr = lora_manager.LoRAManager([p1, p2], pipe)
    sites = [m for m in pipe.unet.modules() if type(m).__name__ == "LoraInjectedLinear"]
    assert sites and all(m.lora_down.weight.shape[0] == 6 for m in sites)
    assert len(pipe.tokenizer) == te.get_input_embeddings().weight.shape[0]   # resized to hold 3 tokens
    mgr.tune([0.25, 2.0])
    want = torch.tensor([0.25] * 4 + [2.0] * 2)
    assert all(torch.equal(m.selector.weight.data.diagonal().cpu().float(), want) for m in sites)
    assert mgr.prompt("a <1> and <2>") == "a <s0-0> and <s1-0><s1-1>"
    with pytest.raises(AssertionError):
        mgr.tune([1.0])


# -------------------------------------------------------------------------------------- lora_add
def test_add_lpl_safetensors_blends_factors_and_keeps_embeddings(tmp_path):
    p1 = _make_lora_file(str(tmp_path / "a.safetensors"), 7, 4, with_tokens=("<a>",))
    p2 = _make_lora_file(str(tmp_path / "b.safetensors"), 8, 4, with_tokens=("<b>",))
    out = str(tmp_path / "o.safetensors")
    lora_add.add(p1, p2, out, alpha_1=0.3, alpha_2=0.9, mode="lpl")
    (t1, m1), (t2, m2), (to, mo) = _read(p1), _read(p2), _read(out)
    assert set(to) == set(t1) | set(t2)
    for k in to:
        if k.startswith(("unet", "text_encoder")):
            assert torch.equal(to[k], 0.3 * t1[k] + 0.9 * t2[k])
    assert torch.equal(to["<a>"], t1["<a>"]) and torch.equal(to["<b>"], t2["<b>"])
    assert mo == {**m1, **m2}


def test_add_lpl_pt_and_text_encoder_companion(tmp_path):
    g = torch.Generator().manual_seed(0)
    mk = lambda: [torch.nn.Parameter(torch.randn(6, 4, generator=g)) if i % 2 == 0 else
                  torch.nn.Parameter(torch.randn(4, 8, generator=g)) for i in range(6)]
    a, b, ta, tb = mk(), mk(), mk(), mk()
    pa, pb, po = (str(tmp_path / n) for n in ("a.pt", "b.pt", "o.pt"))
    torch.save(a, pa), torch.save(b, pb)
    torch.save(ta, L._text_lora_path(pa)), torch.save(tb, L._text_lora_path(pb))
    lora_add.add(pa, pb, po, 0.5, 0.25, mode="lpl", with_text_lora=True)
    o = torch.load(po)
    assert len(o) == 6 and all(torch.equal(x.data, 0.5 * y.data + 0.25 * z.data) for x, y, z in zip(o, a, b))
    ot = torch.load(L._text_lora_path(po))
    assert all(torch.equal(x.data, 0.5 * y.data + 0.25 * z.data) for x, y, z in zip(ot, ta, tb))
    # without the companion on one side: the unet file is still written, the text one skipped
    os.remove(L._text_lora_path(pb))
    po2 = str(tmp_path / "o2.pt")
    lora_add.add(pa, pb, po2, mode="lpl", with_text_lora=True)
    assert os.path.exists(po2) and not os.path.exists(L._text_lora_path(po2))


def test_add_ljl_writes_the_join_and_rejects_unknown_modes(tmp_path):
    p1 = _make_lora_file(str(tmp_path / "a.safetensors"), 9, 4)
    p2 = _make_lora_file(str(tmp_path / "b.safetensors"), 10, 4)
    out = str(tmp_path / "j.safetensors")
    lora_add.add(p1, p2, out, mode="ljl")
    to, mo = _read(out)
    assert all(v.shape[0 if k.endswith("down") else 1] == 8 for k, v in to.items())
    assert all(v == "8" for k, v in mo.items() if k.endswith("rank"))
    with pytest.raises(ValueError):
        lora_add.add(p1, p2, out, mode="nope")
    with pytest.raises(AssertionError):
        lora_add.add(p1, "x.pt", out, mode="ljl")


def test_add_equals_reference_on_files(G, tmp_path):
    p1 = _make_lora_file(str(tmp_path / "a.safetensors"), 11, 4, with_tokens=("<a>",))
    p2 = _make_lora_file(str(tmp_path / "b.safetensors"), 12, 4, with_tokens=("<b>",))
    for mode in ("lpl", "ljl"):
        o = str(tmp_path / f"o_{mode}.safetensors")
        lora_add.add(p1, p2, o, 0.7, 0.4, mode=mode)
        to, mo = _read(o)
        ref = G["add"][mode]
        assert canon_metadata(mo) == ref["metadata"] and to.keys() == ref["tensors"].keys()
        assert {k: digest(v) for k, v in to.items()} == ref["tensors"]


def test_merge_into_pipeline_folds_the_branch_and_restores_plain_modules(tmp_path):
    p = _make_lora_file(str(tmp_path / "a.safetensors"), 13, 4, with_tokens=("<a>",))
    torch.manual_seed(0)
    te = build_text_encoder(tiny=True)
    pipe = types.SimpleNamespace(unet=UNet2DConditionModel(UNetConfig.tiny()), text_encoder=te,
                                 tokenizer=_Tok(te.get_input_embeddings().weight.shape[0]))
    before = {n: w.detach().clone() for n, w in pipe.unet.named_parameters()}
    tok = lora_add.merge_lora_into_pipeline(pipe, p, alpha=0.5, patch_ti=False)
    assert set(tok) == {"<a>"}
    assert not [m for m in pipe.unet.modules() if type(m).__name__.startswith("LoraInjected")]
    after = dict(pipe.unet.named_parameters())
    assert after.keys() == before.keys()
    t, _ = _read(p)
    changed = [n for n in before if not torch.equal(before[n], after[n])]
    assert len(changed) == sum(1 for k in t if k.startswith("unet") and k.endswith(":up"))
    # first site in injection order: W' = W + 0.5 * up @ down
    from lora_b200.inject import _find_modules
    fresh = UNet2DConditionModel(UNetConfig.tiny())          # structure only: which Linear is site 0
    parent, name, child = next(iter(_find_modules(fresh, L.UNET_DEFAULT_TARGET_REPLACE, search_class=[torch.nn.Linear])))
    full = [n for n, m in fresh.named_modules() if m is child][0]
    want = before[full + ".weight"] + 0.5 * (t["unet:0:up"].float() @ t["unet:0:down"].float())
    assert torch.allclose(after[full + ".weight"], want, atol=1e-6)


def test_upl_without_diffusers_fails_loudly(tmp_path):
    with pytest.raises(ImportError):
        lora_add.add("some/dir", "x.safetensors", str(tmp_path / "o"), mode="upl")


# ---------------------------------------------------------------------------- pt -> safetensors
def test_pt_to_safetensors_names_models_from_paths_and_applies_overrides(tmp_path):
    g = torch.Generator().manual_seed(0)
    pairs = lambda r: [torch.randn(8, r, generator=g) if i % 2 == 0 else torch.randn(r, 8, generator=g)
                       for i in range(4)]
    pu, pt_, pe = (str(tmp_path / n) for n in ("w.pt", "w.text_encoder.pt", "w.ti.pt"))
    u, t = pairs(4), pairs(2)
    torch.save(u, pu), torch.save(t, pt_), torch.save({"<tok>": torch.randn(16, generator=g)}, pe)
    out = str(tmp_path / "w.safetensors")
    pt_to_safetensors.convert(pu, pt_, pe, outpath=out, **{"text_encoder.rank": 2})
    ts, meta = _read(out)
    assert torch.equal(ts["unet:0:up"], u[0]) and torch.equal(ts["unet:1:down"], u[3])
    assert torch.equal(ts["text_encoder:1:up"], t[2])
    assert meta["unet:0:rank"] == "4" and meta["text_encoder:1:rank"] == "2" and meta["<tok>"] == "<embed>"
    import json
    assert set(json.loads(meta["text_encoder"])) == L.TEXT_ENCODER_DEFAULT_TARGET_REPLACE
    with pytest.raises(ValueError):
        pt_to_safetensors.convert(pu, outpath=out)
    pt_to_safetensors.convert(pu, outpath=out, overwrite=True)
    # round trip through the loader
    f = safe_open(out, framework="pt", device="cpu")
    parsed = L.parse_safeloras(f)
    assert list(parsed) == ["unet"] and parsed["unet"][1] == [4, 4]


# --------------------------------------------------------------------------- diffusers -> .ckpt
def _vae_keys():
    """Key set of a diffusers AutoencoderKL (SD1.x, pre-0.15 attention names) - structure only."""
    ks = []
    def res(p, shortcut=False):
        for n in ("norm1", "conv1", "norm2", "conv2") + (("conv_shortcut",) if shortcut else ()):
            ks.extend([f"{p}.{n}.weight", f"{p}.{n}.bias"])
    for coder in ("encoder", "decoder"):
        ks += [f"{coder}.conv_in.weight", f"{coder}.conv_in.bias", f"{coder}.conv_out.weight",
               f"{coder}.conv_out.bias", f"{coder}.conv_norm_out.weight", f"{coder}.conv_norm_out.bias"]
        for j in range(2):
            res(f"{coder}.mid_block.resnets.{j}")
        for n in ("group_norm", "query", "key", "value", "proj_attn"):
            ks += [f"{coder}.mid_block.attentions.0.{n}.weight", f"{coder}.mid_block.attentions.0.{n}.bias"]
    for i in range(4):
        for j in range(2):
            res(f"encoder.down_blocks.{i}.resnets.{j}", shortcut=(j == 0 and i in (1, 2)))
        for j in range(3):
            res(f"decoder.up_blocks.{i}.resnets.{j}", shortcut=(j == 0 and i in (2, 3)))
        if i < 3:
            ks += [f"encoder.down_blocks.{i}.downsamplers.0.conv.weight", f"encoder.down_blocks.{i}.downsamplers.0.conv.bias",
                   f"decoder.up_blocks.{i}.upsamplers.0.conv.weight", f"decoder.up_blocks.{i}.upsamplers.0.conv.bias"]
    ks += ["quant_conv.weight", "quant_conv.bias", "post_quant_conv.weight", "post_quant_conv.bias"]
    return ks


def test_unet_key_conversion_known_answers():
    kat = {
        "time_embedding.linear_2.bias": "time_embed.2.bias",
        "conv_in.weight": "input_blocks.0.0.weight",
        "conv_norm_out.bias": "out.0.bias",
        "down_blocks.0.resnets.1.time_emb_proj.weight": "input_blocks.2.0.emb_layers.1.weight",
        "down_blocks.2.attentions.0.transformer_blocks.0.attn2.to_k.weight":
            "input_blocks.7.1.transformer_blocks.0.attn2.to_k.weight",
        "down_blocks.1.downsamplers.0.conv.bias": "input_blocks.6.0.op.bias",
        "down_blocks.3.resnets.0.conv2.weight": "input_blocks.10.0.out_layers.3.weight",
        "mid_block.attentions.0.proj_in.weight": "middle_block.1.proj_in.weight",
        "mid_block.resnets.1.norm1.weight": "middle_block.2.in_layers.0.weight",
        "up_blocks.0.upsamplers.0.conv.weight": "output_blocks.2.1.conv.weight",
        "up_blocks.2.upsamplers.0.conv.weight": "output_blocks.8.2.conv.weight",
        "up_blocks.3.resnets.2.conv_shortcut.weight": "output_blocks.11.0.skip_connection.weight",
        "up_blocks.1.attentions.2.norm.weight": "output_blocks.5.1.norm.weight",
    }
    got = to_ckpt.convert_unet_state_dict({k: i for i, k in enumerate(kat)})
    assert list(got) == list(kat.values())


def test_ckpt_key_conversion_equals_reference(G):
    unet_sd = {k: torch.zeros(1) for k in UNet2DConditionModel(UNetConfig.tiny()).state_dict()}
    assert len(unet_sd) > 300
    ours = to_ckpt.convert_unet_state_dict(dict(unet_sd))
    assert list(ours) == G["ckpt_unet_keys"]
    vae_sd = {k: (torch.zeros(4, 4) if ".attentions.0." in k and k.endswith("weight") and "group_norm" not in k
                  else torch.zeros(4)) for k in _vae_keys()}
    ours = to_ckpt.convert_vae_state_dict(dict(vae_sd))
    assert [[k, list(v.shape)] for k, v in ours.items()] == G["ckpt_vae"]
    assert ours["encoder.mid.attn_1.q.weight"].shape == (4, 4, 1, 1)
    assert "decoder.up.3.block.0.norm1.weight" in ours and "decoder.up.0.upsample.conv.weight" not in ours


def test_convert_to_ckpt_writes_prefixed_half_state_dict(tmp_path):
    root = tmp_path / "pipe"
    for sub in ("unet", "vae", "text_encoder"):
        (root / sub).mkdir(parents=True)
    torch.save({"conv_in.weight": torch.ones(2, 2), "mid_block.resnets.0.conv1.bias": torch.ones(2)},
               root / "unet" / "diffusion_pytorch_model.bin")
    save_file({"encoder.mid_block.attentions.0.query.weight": torch.ones(3, 3),
               "decoder.up_blocks.0.resnets.2.conv_shortcut.bias": torch.ones(3)},
              str(root / "vae" / "diffusion_pytorch_model.safetensors"))
    torch.save({"text_model.final_layer_norm.weight": torch.ones(5)}, root / "text_encoder" / "pytorch_model.bin")
    out = str(tmp_path / "m.ckpt")
    to_ckpt.convert_to_ckpt(str(root), out, as_half=True)
    sd = torch.load(out)["state_dict"]
    assert set(sd) == {"model.diffusion_model.input_blocks.0.0.weight",
                       "model.diffusion_model.middle_block.0.in_layers.2.bias",
                       "first_stage_model.encoder.mid.attn_1.q.weight",
                       "first_stage_model.decoder.up.3.block.2.nin_shortcut.bias",
                       "cond_stage_model.transformer.text_model.final_layer_norm.weight"}
    assert all(v.dtype == torch.float16 for v in sd.values())
    assert sd["first_stage_model.encoder.mid.attn_1.q.weight"].shape == (3, 3, 1, 1)
    with pytest.raises(FileNotFoundError):
        to_ckpt.convert_to_ckpt(str(tmp_path / "nowhere"), out, as_half=False)
