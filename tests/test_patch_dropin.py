"""The reference's ``replace_*()`` start-up mechanism (inference.py:10-24) pointed at the B200 classes: after
``replace_*_b200()`` every reference module that holds one of the replaced classes holds the B200 class instead, and a
state dict saved from the unpatched reference loads into the B200 modules with ``strict=True``.  CPU-only
(construction + state-dict load; compute needs the GPU).  The reference modules are stood in for by empty modules
under the same names, holding the same bindings; the reference checkpoint layouts come from
tests/golden/reference_layouts.npz (make_golden.make_layouts)."""
import sys
import types

import torch

from tests.golden.make_golden import LLAMA_TINY, MMFSNET_TINY, load_layout

_REF = "mm_interleaved.models"
_LLAMA_CLASSES = ("LlamaRMSNorm", "LlamaMLP", "LlamaAttention", "LlamaMMFSAttention", "LlamaDecoderLayer")


def _stand_in_reference(monkeypatch):
    """Modules named like the reference's, each binding its own placeholder classes; the MMFS class is bound a second
    time where the reference imports it (``from ..modules import MMFS`` in ops/modules/__init__.py and sd_mmfs.py)."""
    def module(name, **attrs):
        mod = types.ModuleType(f"{_REF}.{name}")
        for k, v in attrs.items():
            setattr(mod, k, v)
        monkeypatch.setitem(sys.modules, mod.__name__, mod)
        return mod

    mmfs_cls = type("MMFS", (torch.nn.Module,), {})
    return types.SimpleNamespace(
        func=module("utils.ops.functions.ms_deform_attn_func", MSDA=types.ModuleType("MultiScaleDeformableAttention")),
        mmfs=module("utils.ops.modules.mmfs", MMFS=mmfs_cls),
        modules=module("utils.ops.modules", MMFS=mmfs_cls),
        llama=module("decoders.modeling_llama_mmfs", **{n: type(n, (torch.nn.Module,), {}) for n in _LLAMA_CLASSES}),
        sd_mmfs=module("decoders.sd_mmfs", MMFS=mmfs_cls, MMFSNet=type("MMFSNet", (torch.nn.Module,), {}),
                       MMFSBlock=type("MMFSBlock", (torch.nn.Module,), {})))


def _reference_checkpoint(tag):
    return {k: torch.zeros(shape) for k, shape in load_layout(tag).items()}


def test_replace_functions_rebind_the_reference_and_checkpoints_load(monkeypatch):
    import mm_interleaved_b200 as b200
    from mm_interleaved_b200 import patch
    ns = _stand_in_reference(monkeypatch)
    ref_mmfs_cls, ref_layer_cls, ref_net_cls = ns.mmfs.MMFS, ns.llama.LlamaDecoderLayer, ns.sd_mmfs.MMFSNet
    ref_msda = ns.func.MSDA
    try:
        b200.replace_mmfs_b200()
        assert ns.mmfs.MMFS is b200.MMFS and ns.sd_mmfs.MMFS is b200.MMFS and ns.modules.MMFS is b200.MMFS
        assert sys.modules["MultiScaleDeformableAttention"].ms_deform_attn_forward is b200.ms_deform_attn_forward
        assert ns.func.MSDA is sys.modules["MultiScaleDeformableAttention"]

        b200.replace_llama_b200()
        for name in _LLAMA_CLASSES:
            assert getattr(ns.llama, name) is getattr(b200, name)

        b200.replace_visual_b200()
        assert ns.sd_mmfs.MMFSNet is b200.MMFSNet and ns.sd_mmfs.MMFSBlock is b200.MMFSBlock

        b200.replace_all_b200()                                           # idempotent
        assert ns.llama.LlamaDecoderLayer is b200.LlamaDecoderLayer and ns.mmfs.MMFS is b200.MMFS
    finally:
        patch.restore_reference()
    assert ns.mmfs.MMFS is ref_mmfs_cls and ns.sd_mmfs.MMFS is ref_mmfs_cls and ns.llama.LlamaDecoderLayer is ref_layer_cls
    assert ns.sd_mmfs.MMFSNet is ref_net_cls and ns.func.MSDA is ref_msda
    assert "MultiScaleDeformableAttention" not in sys.modules or \
        not getattr(sys.modules["MultiScaleDeformableAttention"], "_b200_dropin", False)

    # checkpoints saved from the unpatched reference load into the B200 modules unchanged
    model = b200.LlamaModel(b200.LlamaMMFSConfig(**LLAMA_TINY))
    assert all(type(l) is b200.LlamaDecoderLayer for l in model.layers)
    assert type(model.layers[0].llama_cross_attn.attn) is b200.MMFS and type(model.norm) is b200.LlamaRMSNorm
    ref_sd = _reference_checkpoint("llama")
    missing, unexpected = model.load_state_dict(ref_sd, strict=True)
    assert not missing and not unexpected
    assert set(model.state_dict().keys()) == set(ref_sd.keys())
    xattn = model.layers[0].llama_cross_attn
    xattn.load_state_dict({k[len("layers.0.llama_cross_attn."):]: v for k, v in ref_sd.items()
                           if k.startswith("layers.0.llama_cross_attn.")}, strict=True)
    b200.MMFSNet(**MMFSNET_TINY).load_state_dict(_reference_checkpoint("mmfsnet"), strict=True)


def test_b200_top_level_model_keeps_the_reference_state_dict_layout():
    """``MMInterleaved`` (B200) exposes the reference's parameter names for the parts whose reference classes import
    here (decoder + text head + glue): every key of the reference ``LlamaModel`` / ``TextDecoder`` layout exists."""
    import pytest
    import mm_interleaved_b200 as b200
    ref_keys = {"mm_decoder." + k for k in load_layout("llama")}
    tiny_vt = dict(clip_config=b200.visual_tokenizer.CLIPVisionConfigLite(hidden_size=64, intermediate_size=128,
                                                                        num_hidden_layers=4, num_attention_heads=4,
                                                                        image_size=32, patch_size=8),
                   perceiver_config=dict(num_queries=3, hidden_size=48, encoder_hidden_size=64, num_hidden_layers=2,
                                         num_attention_heads=4, intermediate_size=96, cross_attention_frequency=1,
                                         qk_normalization=True), grid_size=4)
    try:
        model = b200.MMInterleaved(llm_config=dict(LLAMA_TINY, vocab_size=62), txt_vocab_size=64, seq_len=32,
                                   visual_tokenizer_config=tiny_vt, image_embed_dim=LLAMA_TINY["image_embed_dim"],
                                   cross_attention_frequency=2, spatial_shapes=LLAMA_TINY["spatial_shapes"])
    except Exception as e:                                                # tiny tokenizer dims unsupported on this build
        pytest.skip(f"tiny visual tokenizer config not constructible: {e}")
    keys = set(model.state_dict().keys())
    assert ref_keys <= keys, sorted(ref_keys - keys)[:5]
    for k in ("text_decoder.head.weight", "text_decoder.head.bias", "text_decoder.head_new.weight",
              "text_decoder.head_new.bias", "soi_token", "context_feat_proj.weight", "context_feat_proj.bias"):
        assert k in keys, k
    assert model.text_decoder.head.weight.shape[0] == 64 and model.text_decoder.head_new.weight.shape[0] == 2
    assert any(k.startswith("visual_tokenizer.encoder.") for k in keys)
