"""Generate the committed golden fixtures from the UNMODIFIED reference, executed in the build
container (``/root/reference`` is absent on the GPU box, so the vectors travel instead).

    python tests/golden/make_golden.py            # writes tests/golden/*.npz
    python tests/golden/make_golden.py ref_cuda   # on a B200 after build(): msda_ref_cuda_sampled.npz

The reference ships no golden vectors for this path (SURVEY.md section 4: the pickle that
ops/tests/compare_with_data.py:112-114 expects is not in the repository), so these fixtures
are outputs of the reference's own code run here:

  msda_core_*.npz   ms_deform_attn_core_pytorch (ops/functions/ms_deform_attn_func.py:47-67),
                    fp32 and fp64, on seeded inputs that are stored alongside the outputs
  oracle_msda_loc_modes.npz, oracle_mmfs_seeded.npz, sincos_1d.npz, reference_layouts.npz
                    ("reference_checks"): core / MMFS outputs, sin-cos tables and checkpoint layouts
  msda_ref_cuda_sampled.npz
                    ("ref_cuda"): the reference's own CUDA forward / backward (oracle/_ref/) on a B200
"""
from __future__ import annotations

import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import make_msda_inputs  # noqa: E402
from oracle import ref_loader  # noqa: E402

# name -> (N, spatial_shapes, M, D, Lq, P, seed, loc_mode)
MSDA_CASES = {
    # the reference test-script shape (ops/tests/forward_backward_error.py:175-206)
    "ref_script": (1, [(6, 4), (3, 2)], 2, 64, 2, 2, 0, "uniform"),
    "tiny_edges": (2, [(8, 8), (4, 6), (3, 2)], 4, 32, 37, 4, 1, "edges"),
    "llm_like": (1, [(32, 32), (16, 16), (8, 8)] * 2, 16, 64, 24, 8, 2, "clustered"),
    "sd_like": (1, [(64, 64), (32, 32), (16, 16), (8, 8)], 16, 64, 16, 8, 3, "uniform"),
    "adapter_like": (2, [(16, 16)], 16, 32, 40, 4, 4, "clustered"),
    "odd_dims": (1, [(5, 7), (2, 3)], 3, 24, 9, 3, 5, "edges"),
}


def input_digest(value, loc, attn) -> str:
    import hashlib
    h = hashlib.sha1()
    for t in (value, loc, attn):
        h.update(t.contiguous().numpy().tobytes())
    return h.hexdigest()


def main():
    ref = ref_loader.load()
    core = ref.func.ms_deform_attn_core_pytorch
    for name, (N, shapes, M, D, Lq, P, seed, mode) in MSDA_CASES.items():
        value, ss, starts, loc, attn = make_msda_inputs(N, shapes, M, D, Lq, P, seed=seed, loc_mode=mode)
        out32 = core(value, ss, loc, attn)
        out64 = core(value.double(), ss, loc.double(), attn.double())
        path = os.path.join(HERE, f"msda_core_{name}.npz")
        arrays = dict(spatial_shapes=ss.numpy(), level_start_index=starts.numpy(),
                      out_fp32=out32.numpy(), out_fp64=out64.numpy(),
                      params=np.array([N, M, D, Lq, P, seed], dtype=np.int64), loc_mode=np.array(mode),
                      input_sha1=np.array(input_digest(value, loc, attn)))
        if value.numel() + loc.numel() + attn.numel() <= 200_000:
            # small cases carry their inputs; large ones are regenerated from the seed by
            # oracle.make_msda_inputs and verified against input_sha1
            arrays.update(value=value.numpy(), sampling_loc=loc.numpy(), attn_weight=attn.numpy())
        np.savez_compressed(path, **arrays)
        print(f"{path}: {os.path.getsize(path) / 1024:.0f} KiB  out {tuple(out32.shape)}")


# ---------------------------------------------------------------------------------------------
# MMFS module (ops/modules/mmfs.py:120-276) executed with the reference's own PyTorch core
# ---------------------------------------------------------------------------------------------
# name -> dict(ctor kwargs, N, Lq, n_img, mask kind, ref kind)
MMFS_CASES = {
    # LLM flavour: reference point (0.5,0.5), per-token 3-D mask with causal image visibility
    "llm_tiny": dict(ctor=dict(d_model=192, d_query=192, d_value=128, d_out=192, n_levels=3, n_heads=2, n_points=8,
                               ratio=128 / 192, spatial_shapes=[8, 4, 2], base_spatial_shape=4),
                     N=2, Lq=19, n_img=3, mask="3d", ref="center", seed=0),
    # decode step: Lq = 1 while the mask still has the prefill length -> last row is used (mmfs.py:161-162)
    "llm_decode": dict(ctor=dict(d_model=192, d_query=192, d_value=128, d_out=192, n_levels=3, n_heads=2, n_points=8,
                                 ratio=128 / 192, spatial_shapes=[8, 4, 2], base_spatial_shape=4),
                       N=2, Lq=1, n_img=3, mask="3d_long", ref="center", seed=1),
    # SD flavour: pixel-centre reference grid, 2-D mask, 4 levels, 1 conditioning image, D = 32
    "sd_tiny": dict(ctor=dict(d_model=128, d_query=96, d_value=128, d_out=96, n_levels=4, n_heads=4, n_points=8,
                              ratio=1.0, spatial_shapes=[8, 4, 2, 1], base_spatial_shape=4),
                    N=2, Lq=16, n_img=1, mask="2d", ref="grid", seed=2),
    # 2-D mask with a fully masked sample and an odd head size (generic sampler path), 2 images
    "masked_2d": dict(ctor=dict(d_model=96, d_query=80, d_value=48, d_out=80, n_levels=2, n_heads=4, n_points=3,
                                ratio=1.0, spatial_shapes=[6, 3], base_spatial_shape=3),
                      N=3, Lq=7, n_img=2, mask="2d_masked", ref="center", seed=3),
}


def mmfs_case_inputs(case):
    c = case["ctor"]
    g = torch.Generator().manual_seed(1000 + case["seed"])
    N, Lq, n_img = case["N"], case["Lq"], case["n_img"]
    hw = sum(s * s for s in c["spatial_shapes"])
    query = torch.randn((N, Lq, c["d_query"]), generator=g)
    feat = torch.randn((N, n_img, hw, c["d_value"]), generator=g)
    ss = torch.tensor([(s, s) for s in c["spatial_shapes"]] * n_img, dtype=torch.long)
    starts = torch.cat((ss.new_zeros((1,)), ss.prod(1).cumsum(0)[:-1]))
    if case["mask"] == "3d":
        mask = (torch.rand((N, Lq, n_img), generator=g) < 0.6).float()
        mask[0, 0] = 0                                   # a token that sees no image at all
        mask[1, -1] = 1
    elif case["mask"] == "3d_long":
        mask = (torch.rand((N, 11, n_img), generator=g) < 0.6).float()
        mask[0, -1] = torch.tensor([1.0, 0.0, 1.0])
    elif case["mask"] == "2d":
        mask = torch.ones((N, n_img))
    else:
        mask = torch.tensor([[1.0, 1.0], [0.0, 0.0], [0.0, 1.0]])
    if case["ref"] == "center":
        ref = torch.full((1, Lq, 1, 2), 0.5)
    else:
        side = int(Lq ** 0.5)
        ys, xs = torch.meshgrid(torch.arange(side), torch.arange(side), indexing="ij")
        ref = torch.stack([(xs.flatten() + 0.5) / side, (ys.flatten() + 0.5) / side], -1)[None, :, None, :].float()
    return query, ref, feat, ss, starts, mask


def mmfs_case_module(ref_ns, case):
    torch.manual_seed(2000 + case["seed"])
    mod = ref_ns.mmfs.MMFS(**case["ctor"])
    with torch.no_grad():                                 # make every branch observable
        torch.nn.init.normal_(mod.sampling_offsets.weight, std=0.02)
        torch.nn.init.normal_(mod.attention_weights.weight, std=0.05)
        torch.nn.init.normal_(mod.attention_weights.bias, std=0.5)
        torch.nn.init.normal_(mod.dynamic_offset_mask.weight, std=0.05)
        torch.nn.init.normal_(mod.dynamic_offset_mask.bias, std=0.1)
        torch.nn.init.normal_(mod.value_proj.bias, std=0.1)
        torch.nn.init.normal_(mod.output_proj.bias, std=0.1)
        mod.ignore_token.normal_(std=0.3)
    return mod.eval()


def make_mmfs(ref_ns):
    for name, case in MMFS_CASES.items():
        mod = mmfs_case_module(ref_ns, case)
        query, ref, feat, ss, starts, mask = mmfs_case_inputs(case)
        with torch.no_grad():
            out32 = mod(query, ref, feat, ss, starts, None, mask)
            mod64 = mod.double()
            out64 = mod64(query.double(), ref.double(), feat.double(), ss, starts, None, mask.double())
            mod.float()
        arrays = {f"param/{k}": v.float().numpy() for k, v in mod.state_dict().items()}
        arrays.update(query=query.numpy(), reference_points=ref.numpy(), input_flatten=feat.numpy(),
                      spatial_shapes=ss.numpy(), level_start_index=starts.numpy(), attention_mask=mask.numpy(),
                      out_fp32=out32.numpy(), out_fp64=out64.numpy())
        path = os.path.join(HERE, f"mmfs_{name}.npz")
        np.savez_compressed(path, **arrays)
        print(f"{path}: {os.path.getsize(path) / 1024:.0f} KiB  out {tuple(out32.shape)}")


# ---------------------------------------------------------------------------------------------
# Llama-MMFS decoder (decoders/modeling_llama_mmfs.py) -- tiny configuration, seeded weights
# ---------------------------------------------------------------------------------------------
LLAMA_TINY = dict(vocab_size=64, hidden_size=256, intermediate_size=512, num_hidden_layers=3, num_attention_heads=2,
                  max_position_embeddings=64, rms_norm_eps=1e-6, pad_token_id=0, cross_attention_frequency=2,
                  spatial_shapes=[8, 4, 2], image_embed_dim=512)


def seeded_state_dict(template, seed):
    """Deterministic weights for any module with the reference's parameter names: iterate the names in sorted
    order with one CPU generator.  Used both here (loaded into the reference) and by the tests (loaded
    into the B200 modules), so the multi-MB weights need not be stored in the fixtures."""
    g = torch.Generator().manual_seed(seed)
    out = {}
    for name in sorted(template.keys()):
        t = template[name]
        if not t.is_floating_point():
            out[name] = t.clone()
        elif name.endswith("norm.weight") or name.endswith("layernorm.weight") or ".norm1." in name or ".norm2." in name:
            out[name] = 1.0 + 0.1 * torch.randn(t.shape, generator=g)
        elif name.endswith(".gate"):
            out[name] = torch.full(t.shape, 0.5)
        elif name.endswith("sampling_offsets.bias"):
            out[name] = torch.rand(t.shape, generator=g) * 6 - 3                  # U(-3,3), mmfs.py:103-110
        elif name.endswith("ignore_token"):
            out[name] = torch.zeros(t.shape)
        elif name.endswith(".bias"):
            out[name] = 0.1 * torch.randn(t.shape, generator=g)
        elif name.endswith("embed_tokens.weight") or name.endswith("query_relpos.weight"):
            out[name] = 0.5 * torch.randn(t.shape, generator=g)
        else:
            fan_in = t.shape[-1]
            out[name] = torch.randn(t.shape, generator=g) / (fan_in ** 0.5)
        if name.endswith("sampling_offsets.weight"):
            out[name] = out[name] * 0.3
    return out


def llama_inputs(cfg, B, T, n_img, seed, left_pad=2):
    g = torch.Generator().manual_seed(seed)
    hw = sum(s * s for s in cfg["spatial_shapes"])
    embeds = torch.randn((B, T, cfg["hidden_size"]), generator=g)
    vision = torch.randn((B, n_img, hw, cfg["image_embed_dim"]), generator=g)
    attn_mask = torch.ones((B, T), dtype=torch.long)
    if left_pad and B > 1:
        attn_mask[1, :left_pad] = 0                                    # eval batches are left-padded (collator.py:337)
    position_ids = (attn_mask.cumsum(-1) - 1).clamp(min=0)             # causal_lm_cascade.py:179-185
    cross = (torch.rand((B, T, n_img), generator=g) < 0.6).float()
    cross[0, 0] = 0
    return embeds, vision, attn_mask, position_ids, cross


def make_llama(ref_ns):
    from transformers import LlamaConfig
    cfg = LlamaConfig(**{k: v for k, v in LLAMA_TINY.items() if k not in ("cross_attention_frequency", "spatial_shapes", "image_embed_dim")},
                      hidden_act="silu")
    cfg.cross_attention_frequency = LLAMA_TINY["cross_attention_frequency"]
    cfg.spatial_shapes = LLAMA_TINY["spatial_shapes"]
    cfg.image_embed_dim = LLAMA_TINY["image_embed_dim"]
    model = ref_ns.llama.LlamaModel(cfg).eval()
    sd = seeded_state_dict(model.state_dict(), seed=4242)
    model.load_state_dict(sd)
    B, T, n_img = 2, 12, 2
    embeds, vision, attn_mask, position_ids, cross = llama_inputs(LLAMA_TINY, B, T, n_img, seed=99)
    with torch.no_grad():
        out = model(inputs_embeds=embeds, attention_mask=attn_mask, position_ids=position_ids,
                    vision_hidden_states=vision, cross_attention_mask=cross, use_cache=True, return_dict=True)
        # one decode step on top of the prefill cache (q_len = 1, mask / cross mask grown by one)
        g = torch.Generator().manual_seed(7)
        step = torch.randn((B, 1, LLAMA_TINY["hidden_size"]), generator=g)
        attn2 = torch.cat([attn_mask, torch.ones((B, 1), dtype=torch.long)], 1)
        pos2 = position_ids[:, -1:] + 1
        cross2 = torch.cat([cross, cross[:, -1:]], 1)
        out2 = model(inputs_embeds=step, attention_mask=attn2, position_ids=pos2, past_key_values=out.past_key_values,
                     vision_hidden_states=vision, cross_attention_mask=cross2, use_cache=True, return_dict=True)
        # (no fp64 run: the reference's _make_causal_mask overflows for float64, :28)
    path = os.path.join(HERE, "llama_tiny.npz")
    np.savez_compressed(path, prefill_fp32=out.last_hidden_state.numpy(),
                        decode_fp32=out2.last_hidden_state.numpy(),
                        weight_checksum=np.array(float(sum(v.double().sum() for v in sd.values()))))
    print(f"{path}: {os.path.getsize(path) / 1024:.0f} KiB")


LLAMA_TC = dict(B=2, T=200, n_img=3, seed=123, left_pad=5)      # > 128 rows: two query tiles, four 64-key tiles, padding


def make_llama_tc(ref_ns):
    """The same tiny reference LlamaModel (head_dim 128) on a 200-token prompt: long enough that this repo's 16-bit run
    takes the tcgen05 attention kernel (>= 16 query rows) in every layer, jointly with the fused MMFS sampler.  The
    golden is the reference's fp32 output; the GPU test runs fp16 / bf16 against it (tests/test_llama_gpu.py)."""
    from transformers import LlamaConfig
    cfg = LlamaConfig(**{k: v for k, v in LLAMA_TINY.items() if k not in ("cross_attention_frequency", "spatial_shapes", "image_embed_dim")},
                      hidden_act="silu")
    cfg.max_position_embeddings = 256
    cfg.cross_attention_frequency = LLAMA_TINY["cross_attention_frequency"]
    cfg.spatial_shapes = LLAMA_TINY["spatial_shapes"]
    cfg.image_embed_dim = LLAMA_TINY["image_embed_dim"]
    model = ref_ns.llama.LlamaModel(cfg).eval()
    sd = seeded_state_dict(model.state_dict(), seed=4242)
    model.load_state_dict(sd)
    c = LLAMA_TC
    embeds, vision, attn_mask, position_ids, cross = llama_inputs(LLAMA_TINY, c["B"], c["T"], c["n_img"], seed=c["seed"], left_pad=c["left_pad"])
    with torch.no_grad():
        out = model(inputs_embeds=embeds, attention_mask=attn_mask, position_ids=position_ids,
                    vision_hidden_states=vision, cross_attention_mask=cross, use_cache=False, return_dict=True)
    path = os.path.join(HERE, "llama_tc.npz")
    np.savez_compressed(path, prefill_fp32=out.last_hidden_state.numpy().astype(np.float32),
                        weight_checksum=np.array(float(sum(v.double().sum() for v in sd.values()))))
    print(f"{path}: {os.path.getsize(path) / 1024:.0f} KiB")


# ---------------------------------------------------------------------------------------------
# MMFSNet (decoders/sd_mmfs.py) -- tiny UNet skeleton: 2 resolution stages, 4 skip tensors + mid
# ---------------------------------------------------------------------------------------------
MMFSNET_TINY = dict(input_channel=64, block_out_channels=(32, 64), layers_per_block=1, downsample_factor=8)


def mmfsnet_inputs(seed=11, B=2):
    g = torch.Generator().manual_seed(seed)
    res = [torch.randn((B, 32, 8, 8), generator=g), torch.randn((B, 32, 8, 8), generator=g),
           torch.randn((B, 32, 4, 4), generator=g), torch.randn((B, 64, 4, 4), generator=g)]
    sample = torch.randn((B, 64, 4, 4), generator=g)
    feats = [torch.randn((B, 1, 64, s, s), generator=g) for s in (64, 32, 16, 8)]
    mask = torch.ones((B, 1))
    return sample, res, feats, mask


def mmfsnet_state_dict(template, seed=808):
    sd = seeded_state_dict(template, seed)
    for k in sd:
        if k.endswith("pos_embed"):
            sd[k] = template[k].clone()                         # deterministic sin-cos table
        if k.endswith("conv.weight"):
            sd[k] = sd[k] * 4.0                                  # make the zero-initialised branch observable
    return sd


def make_mmfsnet(ref_ns):
    net = ref_ns.sd_mmfs.MMFSNet(**MMFSNET_TINY).eval()
    sd = mmfsnet_state_dict(net.state_dict())
    net.load_state_dict(sd)
    sample, res, feats, mask = mmfsnet_inputs()
    with torch.no_grad():
        out_sample, out_res = net(sample, res, feats, mask)
    path = os.path.join(HERE, "mmfsnet_tiny.npz")
    arrays = {"sample": out_sample.numpy(), "weight_checksum": np.array(float(sum(v.double().sum() for v in sd.values())))}
    for i, r in enumerate(out_res):
        arrays[f"res{i}"] = r.numpy()
    np.savez_compressed(path, **arrays)
    print(f"{path}: {os.path.getsize(path) / 1024:.0f} KiB")


# ---------------------------------------------------------------------------------------------
# ViT-Adapter building blocks (encoders/vit_adapter/adapter_modules.py): SpatialPriorModule and one
# InteractionBlockWithCls with the two extra extractors; the CLIP blocks in between are replaced by a fixed
# element-wise map so that only reference code under /root/reference is exercised.
# ---------------------------------------------------------------------------------------------
ADAPTER_TINY = dict(dim=256, heads=8, n_points=4, inplanes=16, H=4)     # deform_ratio 0.5 -> head size 16... see below


class _FakeBlocks(torch.nn.Module):
    """Stands in for the sliced CLIPEncoder: x -> tanh(x) * 1.5 (deterministic, parameter-free)."""

    def forward(self, x):
        import types as _t
        return _t.SimpleNamespace(last_hidden_state=torch.tanh(x) * 1.5)


def adapter_inputs(seed=21):
    g = torch.Generator().manual_seed(seed)
    c = ADAPTER_TINY
    H = c["H"]
    img = torch.rand((2, 3, H * 16, H * 16), generator=g)
    x = torch.randn((2, H * H, c["dim"]), generator=g)
    cls = torch.randn((2, 1, c["dim"]), generator=g)
    return img, x, cls


def adapter_state_dict(template, seed):
    sd = seeded_state_dict(template, seed)
    for k in list(sd):
        if k.endswith("gamma"):
            sd[k] = torch.full_like(sd[k], 0.7)                         # injector gamma is zero-initialised
        if k.endswith("sampling_offsets.bias"):
            sd[k] = sd[k] * 0.5
    return sd


def make_adapter(ref_ns):
    ad = ref_ns.adapter
    c = ADAPTER_TINY
    spm = ad.SpatialPriorModule(inplanes=c["inplanes"], embed_dim=c["dim"]).eval()
    blk = ad.InteractionBlockWithCls(dim=c["dim"], num_heads=c["heads"], n_points=c["n_points"], init_values=0.0, drop_path=0.0,
                                     norm_layer=torch.nn.LayerNorm, with_cffn=True, cffn_ratio=0.25, deform_ratio=0.5,
                                     with_cp=False, extra_extractor=True).eval()
    sd_spm = adapter_state_dict(spm.state_dict(), 501)
    sd_blk = adapter_state_dict(blk.state_dict(), 502)
    spm.load_state_dict(sd_spm); blk.load_state_dict(sd_blk)
    img, x, cls = adapter_inputs()
    with torch.no_grad():
        c1, c2, c3, c4 = spm(img)
        d1, d2 = ad.deform_inputs(img)
        cc = torch.cat([c2, c3, c4], dim=1)
        xo, co, clso = blk(x, cc, cls, _FakeBlocks(), d1, d2, c["H"], c["H"])
    path = os.path.join(HERE, "adapter_tiny.npz")
    np.savez_compressed(path, c1=c1.numpy(), c2=c2.numpy(), c3=c3.numpy(), c4=c4.numpy(), x=xo.numpy(), c=co.numpy(),
                        cls=clso.numpy(),
                        checksum=np.array(float(sum(v.double().sum() for v in list(sd_spm.values()) + list(sd_blk.values())))))
    print(f"{path}: {os.path.getsize(path) / 1024:.0f} KiB")


# ---------------------------------------------------------------------------------------------------------
# image-decoder glue: MMInterleaved._prepare_context_features_for_image_decoder / _prepare_mmfs_features_for_image_decoder
# (mm_interleaved.py:254-340).  The module itself does not import under transformers 5.x, so the two method
# definitions are lifted out of the reference FILE with ``ast`` at generation time and executed unmodified against a
# stand-in ``self`` (special_token_dict, seq_len, context_feat_proj) -- nothing of the reference is stored here.
# ---------------------------------------------------------------------------------------------------------
IMGDEC_SOI, IMGDEC_SEQ_LEN, IMGDEC_C = 9, 40, 16


def imgdec_inputs(seed=31):
    g = torch.Generator().manual_seed(seed)
    B, L = 3, 24
    text_ids = torch.randint(10, 50, (B, L), generator=g)
    text_ids[:, 0] = 1
    for r, cols in enumerate([(2, 9, 17), (5,), (3, 20)]):           # <soi> positions per row: 3 + 1 + 2 = 6 images
        for c in cols:
            text_ids[r, c] = IMGDEC_SOI
    n_img = 6
    ctx = torch.randn((B, L, IMGDEC_C), generator=g)
    feats = [torch.randn((n_img, 4, s, s), generator=g) for s in (8, 4, 2)]
    w = torch.randn((IMGDEC_C, IMGDEC_C), generator=g) * 0.3
    b = torch.randn((IMGDEC_C,), generator=g) * 0.1
    nearest_bos = torch.tensor([0, 0, 12, 0, 0, 10])                   # second variant: explicit context starts
    return text_ids, ctx, feats, w, b, nearest_bos


def make_imgdec():
    import ast
    import types
    ref_ns = ref_loader.load()
    path = os.path.join(ref_loader.REF_ROOT, "mm_interleaved", "models", "mm_interleaved.py")
    tree = ast.parse(open(path).read())
    cls = next(n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == "MMInterleaved")
    wanted = {"_prepare_context_features_for_image_decoder", "_prepare_mmfs_features_for_image_decoder"}
    fns = [n for n in cls.body if isinstance(n, ast.FunctionDef) and n.name in wanted]
    assert len(fns) == 2
    mod = ast.Module(body=fns, type_ignores=[])
    from typing import List, Optional
    ns = dict(torch=torch, np=np, List=List, Optional=Optional,
              get_1d_sincos_pos_embed_from_grid=ref_ns.pos_embed.get_1d_sincos_pos_embed_from_grid)
    exec(compile(mod, path, "exec"), ns)
    text_ids, ctx, feats, w, b, nearest_bos = imgdec_inputs()
    proj = torch.nn.Linear(IMGDEC_C, IMGDEC_C)
    with torch.no_grad():
        proj.weight.copy_(w); proj.bias.copy_(b)
    me = types.SimpleNamespace(special_token_dict=dict(soi_token_id=IMGDEC_SOI), seq_len=IMGDEC_SEQ_LEN, context_feat_proj=proj)
    out = {}
    with torch.no_grad():
        for tag, nb in (("a", None), ("b", nearest_bos)):
            cf, cm = ns["_prepare_context_features_for_image_decoder"](me, ctx, text_ids, None, None if nb is None else nb.clone())
            mf, mm = ns["_prepare_mmfs_features_for_image_decoder"](me, feats, text_ids, None if nb is None else nb.clone(),
                                                                   torch.tensor([3, 1, 2]))
            out[f"ctx_{tag}"] = cf.numpy(); out[f"ctx_mask_{tag}"] = cm.numpy(); out[f"mmfs_mask_{tag}"] = mm.numpy()
            for i, f in enumerate(mf):
                out[f"mmfs_{tag}_{i}"] = f.numpy()
    path = os.path.join(HERE, "imgdec_glue.npz")
    np.savez_compressed(path, **out)
    print(f"{path}: {os.path.getsize(path) / 1024:.0f} KiB")


# ---------------------------------------------------------------------------------------------------------
# visual tokenizer: the reference's OWN VisualTokenizer / CLIPVisionTransformerAdapter / CLIPXAttention / qk-norm
# Q-Former attention / PerceiverResampler files (encoders/visual_tokenizer.py:11-101, vit_adapter/vit_adapter_hf.py:36-167,
# vit_adapter/xattn.py:20-141, utils/monkey_patch/blip2_qknorm_monkey_patch.py:8-152, decoders/perceiver.py) executed
# here through oracle/ref_loader.load_visual() -- see its docstring for the three shims (transformers 5.x CLIP / Q-Former
# glue standing in for 4.31, the xformers attention formula, timm.DropPath = Identity).
# ---------------------------------------------------------------------------------------------------------
TOKENIZER_TINY = dict(clip=dict(hidden_size=64, intermediate_size=128, num_hidden_layers=24, num_attention_heads=4,
                                image_size=56, patch_size=14),
                      perceiver=dict(num_queries=5, hidden_size=48, encoder_hidden_size=64, cross_attention_frequency=2,
                                     num_hidden_layers=2, num_attention_heads=4, intermediate_size=96, qk_normalization=True),
                      llm_hidden_size=80, grid_size=4)
QFORMER_TINY = dict(num_queries=8, hidden_size=192, encoder_hidden_size=256, num_hidden_layers=4, num_attention_heads=3,
                    cross_attention_frequency=2, intermediate_size=384, qk_normalization=True)


def tokenizer_state_dict(template, seed=909):
    sd = adapter_state_dict(template, seed)
    g = torch.Generator().manual_seed(seed + 1)
    for k in list(sd):
        if k.endswith("position_ids") or k == "pos_embed":
            sd[k] = template[k].clone()                                  # index buffer / frozen sin-cos table
        elif k.endswith("q_norm.weight") or k.endswith("k_norm.weight") or "layer_norm" in k and k.endswith("weight") \
                or k.endswith("LayerNorm.weight") or k.endswith("_ln.weight") or k.endswith("layrnorm.weight"):
            sd[k] = 1.0 + 0.1 * torch.randn(template[k].shape, generator=g)
        elif k.endswith("proj.weight") and k.count(".") == 1:
            sd[k] = 0.05 * torch.randn(template[k].shape, generator=g)   # 1e-3 init in the reference: make it count
    return sd


def tokenizer_inputs(seed=41):
    return torch.rand((2, 3, 56, 56), generator=torch.Generator().manual_seed(seed))


def qformer_inputs(seed=43):
    g = torch.Generator().manual_seed(seed)
    enc = torch.randn((2, 17, QFORMER_TINY["encoder_hidden_size"]), generator=g)
    mask = torch.ones((2, 17), dtype=torch.long)
    mask[1, 10:] = 0
    return enc, mask


TOKENIZER_FULL = dict(clip=dict(hidden_size=1024, intermediate_size=4096, num_hidden_layers=24, num_attention_heads=16,
                                image_size=224, patch_size=14),
                      perceiver=dict(num_queries=64, hidden_size=768, encoder_hidden_size=1024, cross_attention_frequency=2,
                                     num_hidden_layers=12, num_attention_heads=12, qk_normalization=True),
                      llm_hidden_size=5120, grid_size=16)


def tokenizer_full_inputs(seed=47):
    return torch.rand((1, 3, 224, 224), generator=torch.Generator().manual_seed(seed))


def tokenizer_full_slices(out):
    """The entries of a full-size tokenizer output that the fixture keeps (the outputs are 30 MB): every 8th feature of
    vis_embed / image_embeds, every 16th channel x every 2nd / 4th pixel of the four multi-scale maps."""
    picks = {"vis_embed": out["vis_embed"][..., ::8], "image_embeds": out["image_embeds"][:, ::4, ::8]}
    for i, f in enumerate(out["multiscale_features"]):
        st = 4 if f.shape[-1] >= 32 else 2
        picks[f"ms{i}"] = f[:, ::16, ::st, ::st]
    return picks


def make_tokenizer(full=False):
    from transformers import CLIPVisionConfig
    ns = ref_loader.load_visual()
    c = TOKENIZER_FULL if full else TOKENIZER_TINY
    cfg = CLIPVisionConfig(**c["clip"], hidden_act="quick_gelu", layer_norm_eps=1e-5)
    cfg._attn_implementation = "eager"

    def tiny_encoder(model_path=None, **kw):        # clip_vit_adapter_hf (vit_adapter_hf.py:236-258) minus from_pretrained
        m = ns.vit_adapter.CLIPVisionAdapterModel(cfg)
        ns.xattn.convert_clip_visual_attn(m)
        m.vision_model.set_vis_embed_requires_grad(False)
        return m

    ns.visual_tokenizer.clip_vit_adapter_hf = tiny_encoder
    pc = ref_loader.AttrDict(c["perceiver"], gradient_checkpointing=False, hidden_dropout_prob=0.0,
                             attention_probs_dropout_prob=0.0)
    tok = ns.visual_tokenizer.VisualTokenizer(encoder_model_path="", perceiver_config=pc, llm_hidden_size=c["llm_hidden_size"],
                                              grid_size=c["grid_size"]).eval()
    sd = tokenizer_state_dict(tok.state_dict())
    tok.load_state_dict(sd)
    if full:        # CLIP ViT-L/14 at 224^2 + ViT-Adapter + 12-layer Q-Former, the shapes of the benchmarked step
        with torch.no_grad():
            out = tok(tokenizer_full_inputs())
        path = os.path.join(HERE, "tokenizer_full.npz")
        np.savez_compressed(path, **{k: v.numpy().astype(np.float32) for k, v in tokenizer_full_slices(out).items()},
                            n_keys=np.array(len(sd)), checksum=np.array(float(sum(v.double().sum() for v in sd.values()))))
        print(f"{path}: {os.path.getsize(path) / 1024:.0f} KiB")
        return
    with torch.no_grad():
        out = tok(tokenizer_inputs())
    path = os.path.join(HERE, "tokenizer_tiny.npz")
    np.savez_compressed(path, vis_embed=out["vis_embed"].numpy(), image_embeds=out["image_embeds"].numpy(),
                        **{f"ms{i}": f.numpy() for i, f in enumerate(out["multiscale_features"])},
                        keys=np.array(sorted(sd.keys())),
                        checksum=np.array(float(sum(v.double().sum() for v in sd.values()))))
    print(f"{path}: {os.path.getsize(path) / 1024:.0f} KiB")

    # the Q-Former alone with a key-padding mask (the image decoder's use, decoder_image.py:132-136)
    q = dict(QFORMER_TINY)
    per = ns.perceiver.PerceiverResampler(**q, gradient_checkpointing=False, hidden_dropout_prob=0.0,
                                          attention_probs_dropout_prob=0.0).eval()
    sdq = tokenizer_state_dict(per.state_dict(), seed=919)
    per.load_state_dict(sdq)
    enc, mask = qformer_inputs()
    with torch.no_grad():
        o_mask = per(encoder_hidden_states=enc, encoder_attention_mask=mask, return_dict=False)[0]
        o_nomask = per(encoder_hidden_states=enc, encoder_attention_mask=None, return_dict=False)[0]
    path = os.path.join(HERE, "qformer_qknorm_tiny.npz")
    np.savez_compressed(path, out_masked=o_mask.numpy(), out_unmasked=o_nomask.numpy(), keys=np.array(sorted(sdq.keys())),
                        checksum=np.array(float(sum(v.double().sum() for v in sdq.values()))))
    print(f"{path}: {os.path.getsize(path) / 1024:.0f} KiB")


# ---------------------------------------------------------------------------------------------------------
# Outputs of the reference that the tests used to compute from the reference tree (or from its CUDA op built into
# oracle/_ref/) at test time.  Large outputs are kept as golden_sample(): a fixed, evenly strided subset.
# ---------------------------------------------------------------------------------------------------------
GOLDEN_SAMPLE = 1024


def golden_sample(t, k=GOLDEN_SAMPLE):
    """``k`` evenly strided elements of ``t`` in flat order (all of them if ``t`` is smaller)."""
    flat = t.reshape(-1)
    n = flat.numel()
    return flat if n <= k else flat[torch.arange(k, dtype=torch.long) * n // k]


# ms_deform_attn_core_pytorch on one shape under every location mode: (N, shapes, M, D, Lq, P); seed = mode index
CORE_MODES_CASE = (2, [(12, 10), (6, 5), (3, 3)], 3, 16, 50, 5)
CORE_MODES = ("uniform", "clustered", "edges")


def make_core_modes(ref_ns):
    core = ref_ns.func.ms_deform_attn_core_pytorch
    N, shapes, M, D, Lq, P = CORE_MODES_CASE
    arrays = {}
    for seed, mode in enumerate(CORE_MODES):
        v, s, st, loc, a = make_msda_inputs(N, shapes, M, D, Lq, P, seed=seed, loc_mode=mode)
        arrays[f"{mode}_fp64"] = golden_sample(core(v.double(), s, loc.double(), a.double())).numpy()
        arrays[f"{mode}_fp32"] = golden_sample(core(v, s, loc, a)).numpy()
        arrays[f"{mode}_input_sha1"] = np.array(input_digest(v, loc, a))
    path = os.path.join(HERE, "oracle_msda_loc_modes.npz")
    np.savez_compressed(path, **arrays)
    print(f"{path}: {os.path.getsize(path) / 1024:.0f} KiB")


# the reference MMFS module on a second llm_tiny-shaped case with seeded weights (every branch non-zero)
MMFS_SEEDED = dict(MMFS_CASES["llm_tiny"], seed=77, N=2, Lq=5)


def mmfs_seeded_state_dict(template):
    sd = seeded_state_dict(template, seed=7700)
    sd["ignore_token"] = 0.3 * torch.randn(sd["ignore_token"].shape, generator=torch.Generator().manual_seed(7701))
    return sd


def make_mmfs_seeded(ref_ns):
    case = MMFS_SEEDED
    mod = ref_ns.mmfs.MMFS(**case["ctor"]).eval()
    sd = mmfs_seeded_state_dict(mod.state_dict())
    mod.load_state_dict(sd)
    query, refpts, feat, ss, starts, mask = mmfs_case_inputs(case)
    with torch.no_grad():
        out = mod(query, refpts, feat, ss, starts, None, mask)
    path = os.path.join(HERE, "oracle_mmfs_seeded.npz")
    np.savez_compressed(path, out_fp32=out.numpy(), weight_checksum=np.array(float(sum(v.double().sum() for v in sd.values()))))
    print(f"{path}: {os.path.getsize(path) / 1024:.0f} KiB")


# utils/pos_embed.py get_1d_sincos_pos_embed_from_grid: (embed_dim, positions, rows kept, columns kept)
SINCOS_CASES = ((16, 40, slice(None), slice(None)), (5120, 7, slice(None), slice(None, None, 13)),
                (64, 2048, slice(None, None, 29), slice(None)))


def make_sincos(ref_ns):
    f = ref_ns.pos_embed.get_1d_sincos_pos_embed_from_grid
    arrays = {f"d{dim}_n{n}": f(dim, np.arange(n, dtype=np.float32))[rows, cols] for dim, n, rows, cols in SINCOS_CASES}
    path = os.path.join(HERE, "sincos_1d.npz")
    np.savez_compressed(path, **arrays)
    print(f"{path}: {os.path.getsize(path) / 1024:.0f} KiB")


def ref_llama_config():
    from transformers import LlamaConfig
    extra = ("cross_attention_frequency", "spatial_shapes", "image_embed_dim")
    cfg = LlamaConfig(**{k: v for k, v in LLAMA_TINY.items() if k not in extra}, hidden_act="silu")
    for k in extra:
        setattr(cfg, k, LLAMA_TINY[k])
    return cfg


def make_layouts(ref_ns):
    """Checkpoint layouts (parameter / buffer names and shapes) of the reference LlamaModel (LLAMA_TINY) and MMFSNet
    (MMFSNET_TINY): what a checkpoint saved from the reference holds."""
    arrays = {}
    for tag, mod in (("llama", ref_ns.llama.LlamaModel(ref_llama_config())), ("mmfsnet", ref_ns.sd_mmfs.MMFSNet(**MMFSNET_TINY))):
        sd = mod.state_dict()
        arrays[f"{tag}_keys"] = np.array(list(sd.keys()))
        arrays[f"{tag}_shapes"] = np.array(json.dumps([list(v.shape) for v in sd.values()]))
    path = os.path.join(HERE, "reference_layouts.npz")
    np.savez_compressed(path, **arrays)
    print(f"{path}: {os.path.getsize(path) / 1024:.0f} KiB")


def load_layout(tag):
    z = np.load(os.path.join(HERE, "reference_layouts.npz"))
    return dict(zip([str(k) for k in z[f"{tag}_keys"]], json.loads(str(z[f"{tag}_shapes"]))))


# the reference's own CUDA op (oracle/_ref/, built by oracle/build_ref.py) run on a B200: forward on the cases of
# tests/test_msda_gpu.py::test_against_the_reference_cuda_op, backward on those of test_msda_bwd_gpu.py
REF_CUDA_FWD_CASES, REF_CUDA_FWD_DTYPES = (0, 1, 2, 3, 5), ("float32", "float16", "float64")
REF_CUDA_BWD_DTYPES = ("float32", "float16")


def ref_cuda_fwd_inputs(case, dtype):
    from tests.test_msda_gpu import CASES
    N, shapes, M, D, Lq, P = CASES[case]
    return make_msda_inputs(N, shapes, M, D, Lq, P, seed=300 + case, loc_mode="clustered", dtype=dtype)


def ref_cuda_bwd_inputs(dtype):
    from tests.test_msda_bwd_gpu import CASES
    N, shapes, M, D, Lq, P = CASES[1]
    v, s, st, loc, a = make_msda_inputs(N, shapes, M, D, Lq, P, seed=77, loc_mode="clustered", dtype=dtype)
    go = torch.randn((N, Lq, M * D), generator=torch.Generator().manual_seed(2)).to(dtype)
    return v, s, st, loc, a, go


def make_ref_cuda():
    from oracle import ref_cuda
    ref = ref_cuda.load()
    arrays = {}
    for case in REF_CUDA_FWD_CASES:
        for name in REF_CUDA_FWD_DTYPES:
            dt = getattr(torch, name)
            v, s, st, loc, a = ref_cuda_fwd_inputs(case, dt)
            out = ref.ms_deform_attn_forward(v.to("cuda", dt), s.cuda(), st.cuda(), loc.to("cuda", dt), a.to("cuda", dt), 64)
            arrays[f"fwd{case}_{name}"] = golden_sample(out.cpu()).numpy()
            arrays[f"fwd{case}_{name}_input_sha1"] = np.array(input_digest(v.float(), loc.float(), a.float()))
    for name in REF_CUDA_BWD_DTYPES:
        dt = getattr(torch, name)
        v, s, st, loc, a, go = ref_cuda_bwd_inputs(dt)
        grads = ref.ms_deform_attn_backward(v.to("cuda", dt), s.cuda(), st.cuda(), loc.to("cuda", dt), a.to("cuda", dt),
                                            go.cuda(), 64)
        for g, gname in zip(grads, ("grad_value", "grad_loc", "grad_attn")):
            arrays[f"bwd_{name}_{gname}"] = golden_sample(g.cpu()).numpy()
            arrays[f"bwd_{name}_{gname}_absmax"] = np.array(float(g.float().abs().max()))
        arrays[f"bwd_{name}_input_sha1"] = np.array(input_digest(v.float(), loc.float(), a.float()))
    path = os.path.join(HERE, "msda_ref_cuda_sampled.npz")
    np.savez_compressed(path, **arrays)
    print(f"{path}: {os.path.getsize(path) / 1024:.0f} KiB")


if __name__ == "__main__":
    torch.manual_seed(0)
    which = sys.argv[1:] or ["msda", "mmfs", "llama", "mmfsnet", "adapter", "imgdec", "tokenizer", "reference_checks"]
    if "reference_checks" in which:
        ns = ref_loader.load()
        make_core_modes(ns)
        make_mmfs_seeded(ns)
        make_sincos(ns)
        make_layouts(ns)
    if "ref_cuda" in which:         # needs a GPU and oracle/_ref/
        make_ref_cuda()
    if "tokenizer" in which:
        make_tokenizer()
    if "tokenizer_full" in which:
        make_tokenizer(full=True)
    if "imgdec" in which:
        make_imgdec()
    if "adapter" in which:
        make_adapter(ref_loader.load())
    if "mmfsnet" in which:
        make_mmfsnet(ref_loader.load())
    if "llama" in which:
        make_llama(ref_loader.load())
        make_llama_tc(ref_loader.load())
    if "msda" in which:
        main()
    if "mmfs" in which:
        make_mmfs(ref_loader.load())
