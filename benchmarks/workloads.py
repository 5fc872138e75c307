"""Workloads timed by bench.py.

Each workload owns: seeded synthetic inputs generated on the CPU (so the CPU baseline and the GPU see identical
bits, SURVEY.md 8d), the device-resident step, the end-to-end step through the public API (``MMInterleaved`` with the
reference's batch keys) from pinned host buffers, the per-step result gather, and the roofline / CPU baseline
bookkeeping.  One full-size model (13 B Llama-MMFS decoder + visual tokenizer + SD-2.1 image decoder, random init,
bf16) is built once per process and shared by all workloads.

Unit convention (SURVEY.md 8d): a STEP is one call of the forward hot path on a rank-local batch; ``value`` counts
rank-steps per second over the whole job (world x K / time), so it scales with the number of GPUs under weak scaling;
``sequences_per_s`` (= value x sequences per step) is reported beside it.
"""
from __future__ import annotations

import json
import os
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SOI_ID, IMG_ID, BOS_ID = 32000, 32001, 1       # mm_interleaved.py:33-39 / wds_utils.py:203


def measured_peaks():
    """Roofline denominators: the driver-written MEASURED_PEAKS.json, else the profiling guide's
    stated fallback (6.65 TB/s, 1.59 PFLOP/s)."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": float(d["hbm_gbs"]), "bf16_tflops": float(d["bf16_tflops"]),
                "bf16_tflops_sustained": float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


def ncu_traffic(kernel_key):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch from the committed ``ncu --set full`` capture named in
    profiles/traffic.json ({key: {"bytes_per_launch": ..., "batch": ..., "source": "profiles/<file>"}}); None if absent."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(p):
        return None
    return json.load(open(p)).get(kernel_key)


OUTPUT_SAMPLE = 2 ** 20      # elements kept of an output larger than this (bench.py --dump-outputs)


def output_sample(t, seed=0):
    """``t`` itself, or OUTPUT_SAMPLE of its elements in flat order at fixed seeded positions when it is larger."""
    n = t.numel()
    if n <= OUTPUT_SAMPLE:
        return t
    idx = torch.randint(0, n, (OUTPUT_SAMPLE,), generator=torch.Generator().manual_seed(seed)).sort().values
    return t.reshape(-1)[idx.to(t.device)]


def msda_algorithmic_bytes(N, S, M, D, L, Lq, P, elem_size):
    """SURVEY.md 8d / BASELINE.md section 3: value + loc(2) + weight(1) + out, + shape tables."""
    return elem_size * (N * S * M * D + 3 * N * Lq * M * L * P + N * Lq * M * D) + 24 * L


# ----------------------------------------------------------------------------------------------------------
# the shared full-size model
# ----------------------------------------------------------------------------------------------------------
_MODEL = {}


def full_model(with_image_decoder=True):
    """``MMInterleaved`` at the release dimensions (mm_inference.yaml: Vicuna-13B decoder with MMFS every 4th layer,
    CLIP ViT-L/14 + ViT-Adapter + 64-query Q-Former, SD-2.1-base UNet + MMFSNet + 77-query Q-Former), bf16, seeded
    random init with HF init scales (no network for checkpoints).  Zero-initialised branches of the reference
    (Injector.gamma, MMFSBlock.conv, the gate) get non-zero values so their work is observable."""
    if "m" in _MODEL:
        return _MODEL["m"]
    import mm_interleaved_b200 as m
    from mm_interleaved_b200.mm_interleaved import ImageDecoder
    from mm_interleaved_b200.mmfs import MMFS
    from mm_interleaved_b200.visual_tokenizer import Injector, VisualTokenizer
    dt = torch.bfloat16
    torch.manual_seed(11)
    tok = VisualTokenizer()                                  # ViT-L/14 + adapter + Q-Former(64 queries, 12 layers)
    with torch.no_grad():
        for mod in tok.modules():
            if isinstance(mod, Injector):
                mod.gamma.fill_(0.5)                         # zero-initialised in the reference: make the branch count
        tok.proj.weight.normal_(0.0, 0.02)
    tok = tok.to("cuda", dt).eval()
    with torch.device("meta"):                               # the 13 B decoder is materialised on the GPU directly
        model = m.MMInterleaved(llm_config=m.LlamaMMFSConfig(vocab_size=32000), txt_vocab_size=32002,
                                special_token_dict=dict(bos_token_id=1, eos_token_id=2, pad_token_id=31999,
                                                        soi_token_id=SOI_ID, image_token_id=IMG_ID),
                                visual_tokenizer=tok, image_decoder_config=None)
    for name in ("mm_decoder", "text_decoder", "context_feat_proj"):
        getattr(model, name).to(dt)
    for name in ("mm_decoder", "text_decoder", "context_feat_proj"):
        getattr(model, name).to_empty(device="cuda")
    model.soi_token = torch.nn.Parameter(torch.zeros((1, 5120), dtype=dt, device="cuda"))
    gen = torch.Generator(device="cuda").manual_seed(7)
    with torch.no_grad():
        for name, p in model.named_parameters():
            if name.startswith("visual_tokenizer."):
                continue
            if name.endswith("norm.weight") or name.endswith("layernorm.weight") or ".norm1." in name or ".norm2." in name:
                p.fill_(1.0)
            elif name.endswith(".gate"):
                p.fill_(0.5)
            elif name.endswith("sampling_offsets.bias"):
                p.uniform_(-3.0, 3.0, generator=gen)                     # mmfs.py:103-110
            elif name.endswith("ignore_token") or name.endswith(".bias"):
                p.zero_()
            elif name.endswith("sampling_offsets.weight"):
                p.normal_(0.0, 0.004, generator=gen)
            else:
                p.normal_(0.0, 0.02, generator=gen)
        for mod in model.mm_decoder.modules():
            if isinstance(mod, MMFS):
                mod.scale_ratios = torch.tensor(mod._scale_list, device="cuda")
    if with_image_decoder:
        torch.manual_seed(42)
        dec = ImageDecoder(perceiver_config=dict(num_queries=77, hidden_size=1024, encoder_hidden_size=5120,
                                                 cross_attention_frequency=1, num_hidden_layers=1, num_attention_heads=16),
                           seq_len=77, embed_dim=1024, image_size=512, sd_base_seed=42)      # mm_inference.yaml:18-27
        with torch.no_grad():
            net = dec.decoder.mmfs_module
            for blk in list(net.mmfs_down_blocks) + [net.mmfs_mid_block]:
                blk.conv.weight.normal_(0, 0.02)             # zero-initialised in the reference
        dec = dec.to("cuda", dt).eval()
        dec.decoder.unet.to(memory_format=torch.channels_last)
        model.image_decoder = dec
    model.eval()
    _MODEL["m"] = model
    return model


# ----------------------------------------------------------------------------------------------------------
class Workload:
    metric = "interleaved_steps_per_sec"
    unit = "steps/s"
    dtype_name = "bf16"
    default_steps = None          # secondaries: steps / warm-ups used when run beside the main workload
    default_warmup = 3

    def __init__(self, rank, world, local_batch):
        self.rank, self.world = rank, world
        self.local_batch = local_batch
        self._flush = None
        self._launches = 0
        self._kernel_events = []

    # -- shared helpers -----------------------------------------------------------------
    def flush_l2(self):
        if self._flush is None:
            self._flush = torch.empty(192 * 1024 * 1024, dtype=torch.uint8, device="cuda")  # > 126 MB L2
        self._flush.zero_()

    def reset_counters(self):
        self._launches = 0
        self._kernel_events = []
        from mm_interleaved_b200 import ops
        ops.launch_counter[0] = 0

    def launch_count(self):
        from mm_interleaved_b200 import ops
        return self._launches + ops.launch_counter[0]

    def units_per_step(self):
        return 1                                    # one rank-local step

    def extras(self, value):
        return {}

    def gather(self, dist):
        """One all_gather of the per-rank result checksum per step (the only collective)."""
        if dist is None:
            return
        chk = self.result_checksum()
        out = [torch.empty_like(chk) for _ in range(self.world)]
        dist.all_gather(out, chk)

    def kernel_stats(self):
        torch.cuda.synchronize()
        ms = [a.elapsed_time(b) for a, b in self._kernel_events]
        return {"launches": len(ms), "avg_ms": sum(ms) / len(ms) if ms else None}

    def outputs(self):
        """{name: tensor}: what the last timed step computed, as its caller receives it (bench.py --dump-outputs)."""
        raise NotImplementedError

    def teardown(self):
        pass


def _timed(events_list, fn, count=None):
    """Wrap ``fn`` so that each call is bracketed by CUDA events on the current stream."""
    def wrapper(*a, **k):
        if torch.cuda.is_current_stream_capturing():
            return fn(*a, **k)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = fn(*a, **k)
        e1.record()
        events_list.append((e0, e1))
        if count is not None:
            count[0] += 1
        return r
    return wrapper


class _Patch:
    """Temporarily replace attributes (timing hooks around this repo's kernel wrappers); undone at teardown."""

    def __init__(self):
        self._undo = []

    def set(self, obj, name, new):
        self._undo.append((obj, name, getattr(obj, name)))
        setattr(obj, name, new)

    def restore(self):
        while self._undo:
            obj, name, old = self._undo.pop()
            setattr(obj, name, old)


# ----------------------------------------------------------------------------------------------------------
class MsdaCfg3(Workload):
    """BASELINE cfg 3, deformable-attention sampler only: the 10 MMFS cross-attention layers'
    MSDA launches for `local_batch` 4-image / 2048-token sequences per GPU (per layer: N =
    local_batch, L = 12, S = 5376, Lq = 2048, M = 16, D = 64, P = 8, bf16) through the drop-in op."""

    name = "msda_cfg3"
    LAYERS = 10
    SHAPES = [(32, 32), (16, 16), (8, 8)] * 4
    M, D, Lq, P = 16, 64, 2048, 8

    def make_host_inputs(self, pin):
        from oracle import level_start_index
        B = self.local_batch or 2
        self.B = B
        g = torch.Generator().manual_seed(1234 + self.rank)
        L = len(self.SHAPES)
        shapes = torch.tensor(self.SHAPES, dtype=torch.long)
        self.shapes_h, self.starts_h = shapes, level_start_index(shapes)
        S = int(shapes.prod(1).sum())
        self.S, self.L = S, L
        dt = torch.bfloat16
        self.layers_h = []
        for _ in range(self.LAYERS):
            value = torch.rand((B, S, self.M, self.D), generator=g).to(dt)
            off = (torch.rand((B, self.Lq, self.M, 4, 1, self.P, 2), generator=g) * 6 - 3) / 16.0
            off = off + 0.05 * torch.randn((B, self.Lq, self.M, 4, 1, self.P, 2), generator=g)
            loc = (0.5 + off).expand(B, self.Lq, self.M, 4, 3, self.P, 2).reshape(B, self.Lq, self.M, L, self.P, 2)
            logits = torch.randn((B, self.Lq, self.M, L, self.P), generator=g)
            vis = self.visibility()                                     # (Lq, 4) 0/1
            logits = logits + (1.0 - vis)[None, :, None, :, None].repeat_interleave(3, dim=3) * -10000.0
            attn = torch.softmax(logits.flatten(-2), -1).view(B, self.Lq, self.M, L, self.P)
            lay = tuple(t.to(dt).contiguous() for t in (value, loc, attn))
            self.layers_h.append(tuple(t.pin_memory() for t in lay) if pin else lay)

    def setup(self):
        import mm_interleaved_b200 as m
        self.m = m
        self.make_host_inputs(pin=True)
        B, dt = self.B, torch.bfloat16
        self.shapes_d, self.starts_d = self.shapes_h.cuda(), self.starts_h.cuda()
        self.layers_d = [tuple(t.cuda() for t in lay) for lay in self.layers_h]
        self.out_h = torch.empty((B, self.Lq, self.M * self.D), dtype=dt).pin_memory()
        self.last = None
        self.reset_counters()

    def visibility(self):
        t = torch.arange(self.Lq)
        soi = torch.tensor([1, 512, 1024, 1536]) + 1
        nearest_bos = torch.where(t >= 1023, 1023, 0)
        return ((soi[None, :] > nearest_bos[:, None]) & (soi[None, :] <= t[:, None])).float()

    def extras(self, value):
        return {"sequences_per_step": self.B, "sequences_per_s": value * self.B}

    def step_device(self):
        for (value, loc, attn) in self.layers_d:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            self.last = self.m.ms_deform_attn_forward(value, self.shapes_d, self.starts_d, loc, attn, 64)
            e1.record()
            self._kernel_events.append((e0, e1))
            self._launches += 1

    def step_e2e(self):
        for (value, loc, attn) in self.layers_h:
            self.m.ms_deform_attn_forward_host(value, self.shapes_h, self.starts_h, loc, attn, out=self.out_h)
            self._launches += 1
        self.last = self.out_h

    def result_checksum(self):
        return self.last.float().sum().reshape(1).to("cuda")

    def outputs(self):
        return {"out": output_sample(self.last)}             # the step's last layer

    def h2d_bytes(self):
        return sum(t.numel() * t.element_size() for lay in self.layers_h for t in lay)

    def d2h_bytes(self):
        return self.LAYERS * self.out_h.numel() * self.out_h.element_size()

    def config(self):
        return {"workload": "BASELINE cfg3 MMFS deformable-attention sampler only (drop-in op): 10 cross-attn layers x "
                            f"{self.B} sequences/GPU (L=12,S=5376,Lq=2048,M=16,D=64,P=8)",
                "step_unit": f"the 10 sampler launches of {self.B} sequences", "sequences_per_step": self.B,
                "global_batch": self.B * self.world, "seq_len": 2048, "images_per_seq": 4,
                "parallelism": f"dp{self.world}", "l2": "192 MiB buffer written between timed steps (L2 flush)"}

    def roofline(self, kernel):
        peaks = measured_peaks()
        ab = msda_algorithmic_bytes(self.B, self.S, self.M, self.D, self.L, self.Lq, self.P, 2)
        achieved = ab / (kernel["avg_ms"] * 1e-3) / 1e9 if kernel["avg_ms"] else None
        return {"kernel": "msda_fwd_rows_kernel<bf16,64>", "bound": "hbm", "achieved": achieved,
                "peak": peaks["hbm_gbs"], "peak_source": peaks["source"], "unit": "GB/s",
                "frac": achieved / peaks["hbm_gbs"] if achieved else None,
                "algorithmic_bytes_per_launch": ab, "avg_launch_us": kernel["avg_ms"] * 1e3 if kernel["avg_ms"] else None,
                "launches_timed": kernel["launches"], "traffic": None}

    def cpu_baseline(self):
        from oracle import msda_core_pytorch
        threads = os.cpu_count() or 1
        torch.set_num_threads(threads)
        value, loc, attn = (t[:1].float() for t in self.layers_h[0])
        msda_core_pytorch(value, self.shapes_h, loc, attn)
        t0, n = time.time(), 0
        while n < 3 or time.time() - t0 < 8.0:
            msda_core_pytorch(value, self.shapes_h, loc, attn)
            n += 1
        per_layer = (time.time() - t0) / n
        return {"value": 1.0 / (per_layer * self.LAYERS * self.B), "unit": self.unit, "cores": threads, "kind": "port",
                "sample": f"{n} runs of 1 layer x 1 sequence ({per_layer * 1e3:.0f} ms each), fp32, scaled x{self.LAYERS} layers "
                          f"x {self.B} sequences per step"}

    def setup_cpu_only(self):
        self.make_host_inputs(pin=False)

    def reference_step(self):
        from oracle import msda_core_pytorch
        value, loc, attn = (t[:1].float() for t in self.layers_h[0])
        t0 = time.time()
        msda_core_pytorch(value, self.shapes_h, loc, attn)
        return time.time() - t0

    def reference_value(self, samples):
        per_layer = sum(samples) / len(samples)
        return 1.0 / (per_layer * self.LAYERS * self.B)

    reference_sample = "each sample = 1 of the 10 sampler layers of 1 sequence, fp32, scaled to 10 layers x the step's sequences"


# ----------------------------------------------------------------------------------------------------------
class InterleavedCfg3(Workload):
    """BASELINE cfg 3: the interleaved image-text forward on 4-image / 2048-token sequences, bf16, through the
    reference surface ``MMInterleaved.forward(text_ids, image_tensors, num_image_per_seq)`` (mm_interleaved.py:408-455
    up to the logits): visual tokenizer (CLIP ViT-L/14 + ViT-Adapter + 12-layer Q-Former, visual_tokenizer.py:65-101) on
    the 4 x B images, embed splice + image-visibility mask + MMFS feature packing (:121-252), the 40-layer Llama-13B
    decoder with MMFS cross-attention in every 4th layer (modeling_llama_mmfs.py:623-752), text head
    (decoder_text.py:140-163) and arg-max.  Random-init weights of the real architecture, synthetic token layout of
    SURVEY.md 8d.  Steps ROTATE between distinct image / token sets, so no step can reuse another step's image-side work."""

    name = "interleaved_cfg3"
    T, N_IMG, TOK_PER_IMG = 2048, 4, 64
    SOI_AT = (1, 512, 1024, 1536)
    EXTRA_BOS_AT = (1023,)
    LAYERS_CROSS, LAYERS_TOTAL = 10, 40
    SOI_ID, IMG_ID = SOI_ID, IMG_ID
    DEFAULT_B = 4
    N_SETS = 2
    label = "cfg3"

    def make_host_inputs(self, pin):
        B = self.local_batch or self.DEFAULT_B
        self.B = B
        g = torch.Generator().manual_seed(4321 + self.rank)
        self.host_sets = []
        for _ in range(self.N_SETS):
            ids = torch.randint(3, 31999, (B, self.T), generator=g)
            ids[:, 0] = BOS_ID
            for s in self.SOI_AT:
                ids[:, s] = self.SOI_ID
                ids[:, s + 1:s + 1 + self.TOK_PER_IMG] = self.IMG_ID
            for s in self.EXTRA_BOS_AT:
                ids[:, s] = BOS_ID
            images = torch.rand((B * self.N_IMG, 3, 224, 224), generator=g)      # [0,1] like the reference's image_tensors
            nimg = torch.full((B,), self.N_IMG, dtype=torch.long)
            st = [ids, images, nimg]
            self.host_sets.append([t.pin_memory() for t in st] if pin else st)
        self.host = self.host_sets[0]

    def setup(self):
        from mm_interleaved_b200 import ops, sampler
        import mm_interleaved_b200.llama_mmfs as lm
        import mm_interleaved_b200.mmfs as mmfs_mod
        self.make_host_inputs(pin=True)
        self.model = full_model()
        self.model.enable_cuda_graphs(tokenizer=True)
        self.dev_sets = [[t.cuda() for t in st] for st in self.host_sets]
        self.out_h = torch.empty((self.B, self.T), dtype=torch.long).pin_memory()
        self.last = None
        self._i = 0
        # time the dominant hand-written kernels with CUDA events from inside the step
        self._sampler_events, self._attn_events = [], []
        self._patch = _Patch()
        T = self.T
        orig_attn = ops.attention

        def timed_attn(q, *a, **k):
            if q.shape[1] != T or q.shape[3] != 128 or torch.cuda.is_current_stream_capturing():
                return orig_attn(q, *a, **k)                      # only the Llama prefill attention is the roofline subject
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); r = orig_attn(q, *a, **k); e1.record()
            self._attn_events.append((e0, e1))
            return r

        cnt = [0]
        self._sampler_count = cnt
        self._patch.set(mmfs_mod._sampler, "mmfs_sampler_forward", _timed(self._sampler_events, sampler.mmfs_sampler_forward, cnt))
        self._patch.set(lm.ops, "attention", timed_attn)
        with torch.no_grad():                                     # capture the tokenizer graph, fill weight-derived caches
            self._forward(self.dev_sets[0])
        self.reset_counters()

    def teardown(self):
        self._patch.restore()
        self.last_logits = None

    def reset_counters(self):
        super().reset_counters()
        self._sampler_events.clear()
        self._attn_events.clear()
        self._sampler_count[0] = 0

    def launch_count(self):
        return super().launch_count() + self._sampler_count[0]

    def extras(self, value):
        return {"sequences_per_step": self.B, "sequences_per_s": value * self.B}

    def _forward(self, tensors):
        ids, images, nimg = tensors
        with torch.no_grad():
            out = self.model(text_ids=ids, image_tensors=images, num_image_per_seq=nimg, attention_mask=None,
                             max_num_image=self.N_IMG, return_loss=False)
            self.last_logits = out["text_logits"]
            return self.last_logits.argmax(-1)

    def step_device(self):
        self.last = self._forward(self.dev_sets[self._i % self.N_SETS])
        self._i += 1

    def step_e2e(self):
        host = self.host_sets[self._i % self.N_SETS]
        self._i += 1
        dev = [t.to("cuda", non_blocking=True) for t in host]
        pred = self._forward(dev)
        self.out_h.copy_(pred, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        self.last = pred

    def result_checksum(self):
        return self.last.sum().reshape(1).float()

    def outputs(self):
        return {"text_ids": self.last, "text_logits": output_sample(self.last_logits)}

    def h2d_bytes(self):
        return sum(t.numel() * t.element_size() for t in self.host)

    def d2h_bytes(self):
        return self.out_h.numel() * self.out_h.element_size()

    def kernel_stats(self):
        torch.cuda.synchronize()
        s = [a.elapsed_time(b) for a, b in self._sampler_events]
        t = [a.elapsed_time(b) for a, b in self._attn_events]
        return {"launches": len(s), "avg_ms": sum(s) / len(s) if s else None,
                "attn_launches": len(t), "attn_avg_ms": sum(t) / len(t) if t else None}

    def config(self):
        return {"workload": f"BASELINE {self.label} interleaved forward through MMInterleaved.forward(text_ids, image_tensors, "
                            f"num_image_per_seq): {self.B} sequences/GPU x ({self.N_IMG} images 224^2, {self.T} tokens): visual "
                            "tokenizer (CLIP ViT-L/14 + ViT-Adapter + Q-Former) + embed splice + visibility mask + MMFS feature "
                            "packing + Llama-13B decoder (40 layers, MMFS cross-attn every 4th) + text head + argmax",
                "step_unit": f"one forward call on the rank-local batch of {self.B} sequences", "sequences_per_step": self.B,
                "global_batch": self.B * self.world, "seq_len": self.T, "images_per_seq": self.N_IMG,
                "parallelism": f"dp{self.world}",
                "params": "13B Llama + 10 MMFS layers + 0.45B visual tokenizer (+ 1.3B image decoder resident, unused here), random init, bf16",
                "inputs": f"{self.N_SETS} distinct image/token sets rotated step by step (no cross-step reuse of image-side work)",
                "l2": "192 MiB buffer written between timed steps (L2 flush); weights (27 GB) exceed L2 anyway",
                "cuda_graph": "visual tokenizer captured once per image-batch shape inside MMInterleaved and replayed; decoder eager"}

    def roofline(self, kernel):
        peaks = measured_peaks()
        n_img = self.N_IMG
        S, M, D, L, Lq, P = 1344 * n_img, 16, 64, 3 * n_img, self.T, 8
        ab = msda_algorithmic_bytes(self.B, S, M, D, L, Lq, P, 2)            # SURVEY.md 8d figure (34.1 MB / layer / sequence at cfg 3)
        C = M * P * 2 + M * 3 * (P + 1)
        fused = 2 * (self.B * S * M * D + self.B * Lq * C + 50 * C + self.B * Lq * M * D) + self.B * n_img * Lq
        t = kernel["avg_ms"] * 1e-3 if kernel["avg_ms"] else None
        achieved = ab / t / 1e9 if t else None
        flops = 4.0 * self.B * self.T * self.T * 5120 / 2                     # causal QK^T + PV per layer
        ta = kernel["attn_avg_ms"] * 1e-3 if kernel.get("attn_avg_ms") else None
        tr = ncu_traffic(f"mmfs_sampler_{self.label}")
        return {"kernel": "mmfs_sampler_v2_kernel<bf16,3 levels> (fused MMFS deform-attn sampler)", "bound": "hbm",
                "achieved": achieved, "peak": peaks["hbm_gbs"], "peak_source": peaks["source"], "unit": "GB/s",
                "frac": achieved / peaks["hbm_gbs"] if achieved else None,
                "algorithmic_bytes_per_launch": ab, "fused_kernel_bytes_per_launch": fused,
                "achieved_fused_bytes_GBs": fused / t / 1e9 if t else None,
                "avg_launch_us": t * 1e6 if t else None, "launches_timed": kernel["launches"],
                "traffic": tr["bytes_per_launch"] * self.B / tr["batch"] if tr else None,
                "traffic_source": tr["source"] if tr else None,
                "attention": {"kernel": "attn_fwd_kernel<bf16,128> (tcgen05)", "bound": "tensor",
                              "achieved": flops / ta / 1e12 if ta else None, "peak": peaks["bf16_tflops_sustained"],
                              "unit": "TFLOP/s", "frac": flops / ta / 1e12 / peaks["bf16_tflops_sustained"] if ta else None,
                              "flops_per_launch": flops, "avg_launch_us": ta * 1e6 if ta else None,
                              "launches_timed": kernel.get("attn_launches")}}

    # ---- CPU baseline / reference arm: oracle restatement of the reference forward, bounded sample ----
    def setup_cpu_only(self):
        self.make_host_inputs(pin=False)

    def _cpu_layer_weights(self, cross, seed):
        import mm_interleaved_b200  # noqa: F401  (module definitions only: parameter names / shapes)
        from mm_interleaved_b200.llama_mmfs import LlamaDecoderLayer, LlamaMMFSConfig
        layer = LlamaDecoderLayer(LlamaMMFSConfig(), cross, 0)
        g = torch.Generator().manual_seed(seed)
        sd = {}
        for k, v in layer.state_dict().items():
            if k.endswith("norm.weight") or k.endswith("layernorm.weight") or ".norm1." in k or ".norm2." in k:
                sd["layers.0." + k] = torch.ones_like(v)
            elif k.endswith(".gate"):
                sd["layers.0." + k] = torch.full_like(v, 0.5)
            elif k.endswith("sampling_offsets.bias"):
                sd["layers.0." + k] = torch.rand(v.shape, generator=g) * 6 - 3
            elif k.endswith(".bias") or k.endswith("ignore_token"):
                sd["layers.0." + k] = torch.zeros_like(v)
            else:
                sd["layers.0." + k] = torch.randn(v.shape, generator=g) * 0.02
        return sd

    def reference_step(self):
        """Bounded CPU sample: ONE plain decoder layer + ONE MMFS cross-attention layer of ONE sequence (fp32) through
        the oracle restatement of the reference (oracle/llama.py, oracle/mmfs.py, oracle/glue.py)."""
        from oracle.glue import cross_attention_mask_ref, pack_mmfs_features_ref
        from oracle.llama import additive_mask_ref, llama_layer_ref
        if not hasattr(self, "_cpu"):
            ids = self.host[0][:1]
            nimg = torch.tensor([self.N_IMG])
            x = torch.randn((1, self.T, 5120), generator=torch.Generator().manual_seed(5)) * 0.5
            gf = torch.Generator().manual_seed(9)
            feats = pack_mmfs_features_ref([torch.randn((self.N_IMG, 1024, sz, sz), generator=gf) for sz in (32, 16, 8)],
                                           [32, 16, 8], nimg)
            cross = cross_attention_mask_ref(ids, nimg, BOS_ID, self.SOI_ID)
            cfg = dict(eps=1e-6, n_heads=40, n_layers=1, spatial_shapes=[(32, 32), (16, 16), (8, 8)])
            add_mask = additive_mask_ref(torch.ones((1, self.T)), self.T, 0, torch.float32)
            pos = torch.arange(self.T)[None]
            self._cpu = (x, feats, cross, cfg, add_mask, pos, self._cpu_layer_weights(False, 1), self._cpu_layer_weights(True, 2))
        x, feats, cross, cfg, add_mask, pos, w_plain, w_cross = self._cpu
        with torch.no_grad():
            t0 = time.time()
            llama_layer_ref(w_plain, 0, x, None, None, add_mask, pos, cfg)
            t1 = time.time()
            llama_layer_ref(w_cross, 0, x, feats, cross, add_mask, pos, cfg)
            t2 = time.time()
        return (t1 - t0, t2 - t1)

    def reference_value(self, samples):
        tp = sum(s[0] for s in samples) / len(samples)
        tc = sum(s[1] for s in samples) / len(samples)
        return 1.0 / (self.B * (30 * tp + 10 * tc))

    @property
    def reference_sample(self):
        return (f"each sample = 1 plain + 1 MMFS cross-attention decoder layer of 1 sequence (T={self.T}, {self.N_IMG} images) in fp32 "
                f"through the oracle restatement; step time = {self.B} sequences x (30*t_plain + 10*t_cross); the visual tokenizer, "
                "glue and text head (< 3 % of the FLOPs) are not in the CPU sample (an extrapolation, not a full CPU forward)")

    def cpu_baseline(self):
        threads = min(os.cpu_count() or 1, 64)
        torch.set_num_threads(threads)
        self.reference_step()
        s = [self.reference_step()]
        return {"value": self.reference_value(s), "unit": self.unit, "cores": threads, "kind": "port",
                "sample": f"1 plain layer ({s[0][0]:.2f} s) + 1 MMFS cross layer ({s[0][1]:.2f} s) of 1 sequence, fp32, oracle "
                          f"restatement of the reference forward; scaled to 30 plain + 10 cross layers x {self.B} sequences per step"}


class InterleavedCfg2(InterleavedCfg3):
    """BASELINE cfg 2: CLIP ViT-L/14 encode + Llama-13B prefill, 1-image context, seq_len 512, bf16, one B200
    (the same ``MMInterleaved.forward`` call as cfg 3 on shorter single-image sequences)."""

    name = "interleaved_cfg2"
    T, N_IMG = 512, 1
    SOI_AT = (1,)
    EXTRA_BOS_AT = ()
    DEFAULT_B = 8
    label = "cfg2"
    default_steps, default_warmup = 6, 3


# ----------------------------------------------------------------------------------------------------------
class SdCfg4(Workload):
    """BASELINE cfg 4: SD-2.1 UNet 50-step classifier-free-guidance denoise at 512^2 (latents 64^2) with MMFS
    conditioning on one context image, batch 8 per GPU (16 with CFG), through ``StableDiffusion.generate_images``
    (decoders/sd.py:142-218: DDPM scheduler, seeded generator); a step = one full 50-step denoise of the local batch."""

    name = "sd_cfg4"
    metric = "sd_unet_denoise_steps_per_sec"
    STEPS = 50
    default_steps, default_warmup = 2, 2      # two warm-up loops: graph capture, then both input sets' first-use allocations
    CONV_SHAPE = (1280, 1280, 16, 3)          # Cin, Cout, map side, kernel: the conv timed for the roofline sub-object

    def setup(self):
        from mm_interleaved_b200 import ops, unet_sd
        self.ops, self.unet_sd = ops, unet_sd
        self.B = self.local_batch or 8
        dt = torch.bfloat16
        self.sd = full_model().image_decoder.decoder                       # StableDiffusion: unet + mmfs_module + scheduler
        self.sd.enable_cuda_graphs(True)                                   # one UNet graph, kept across generate_images calls
        g = torch.Generator().manual_seed(42 + self.rank)                  # sd_base_seed: 42 (mm_inference.yaml:23)
        mk = lambda: ([torch.randn((self.B, 4, 64, 64), generator=g), torch.randn((self.B, 77, 1024), generator=g) * 0.02] +
                      [torch.randn((self.B, 1, 1024, s, s), generator=g) for s in (64, 32, 16, 8)])
        self.host_sets = [[t.to(dt).pin_memory() for t in mk()] for _ in range(2)]
        self.host = self.host_sets[0]
        self.dev_sets = [[t.cuda() for t in st] for st in self.host_sets]
        self.mask = torch.ones((self.B, 1), device="cuda")
        self.neg = torch.zeros((self.B, 77, 1024), device="cuda", dtype=dt)
        self.out_h = torch.empty((self.B, 4, 64, 64), dtype=dt).pin_memory()
        self._attn_events, self._conv_events = [], []
        self._i = 0
        self._patch = _Patch()
        orig_attn, orig_conv = ops.attention, ops.conv2d
        cin, cout, side, ks = self.CONV_SHAPE

        def timed_attn(q, kk, *a, **k):
            if q.shape[1] != 4096 or kk.shape[1] != 4096 or torch.cuda.is_current_stream_capturing():
                return orig_attn(q, kk, *a, **k)                    # only the T = 4096 self-attention calls are timed
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); r = orig_attn(q, kk, *a, **k); e1.record()
            self._attn_events.append((e0, e1))
            return r

        def timed_conv(x, w, *a, **k):
            if (x.shape[1] != cin or w.shape[0] != cout or x.shape[2] != side or w.shape[1] != ks
                    or torch.cuda.is_current_stream_capturing()):
                return orig_conv(x, w, *a, **k)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); r = orig_conv(x, w, *a, **k); e1.record()
            self._conv_events.append((e0, e1))
            return r

        self._patch.set(unet_sd.ops, "attention", timed_attn)
        self._patch.set(unet_sd.ops, "conv2d", timed_conv)
        self.reset_counters()

    def teardown(self):
        self._patch.restore()

    def reset_counters(self):
        super().reset_counters()
        self._attn_events.clear()
        self._conv_events.clear()

    def extras(self, value):
        return {"images_per_step": self.B, "images_per_s": value * self.B, "unet_evaluations_per_step": self.STEPS}

    def _run(self, t):
        lat, cond, feats = t[0], t[1], list(t[2:])
        return self.sd.generate_images(text_embeds=cond, negative_prompt_embeds=self.neg, num_inference_steps=self.STEPS,
                                       mini_bs=self.B, guidance_scale=7.5, mmfs_features=feats, mmfs_mask=self.mask, latents=lat)

    def step_device(self):
        self.last = self._run(self.dev_sets[self._i % 2])
        self._i += 1

    def step_e2e(self):
        host = self.host_sets[self._i % 2]
        self._i += 1
        dev = [t.to("cuda", non_blocking=True) for t in host]
        self.last = self._run(dev)
        self.out_h.copy_(self.last, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    def result_checksum(self):
        return self.last.float().sum().reshape(1)

    def outputs(self):
        return {"latents": output_sample(self.last)}

    def h2d_bytes(self):
        return sum(t.numel() * t.element_size() for t in self.host)

    def d2h_bytes(self):
        return self.out_h.numel() * self.out_h.element_size()

    def kernel_stats(self):
        torch.cuda.synchronize()
        if not self._conv_events:
            # the timed steps replayed a CUDA graph (nothing to wrap): time the same kernels in a few EAGER evaluations of
            # the same loop, outside the timed region
            graphs, self.sd._unet_graphs = self.sd._unet_graphs, None
            steps, self.STEPS = self.STEPS, 4
            try:
                self._run(self.dev_sets[0])
            finally:
                self.sd._unet_graphs, self.STEPS = graphs, steps
            torch.cuda.synchronize()
        t = [a.elapsed_time(b) for a, b in self._attn_events]
        c = [a.elapsed_time(b) for a, b in self._conv_events]
        return {"launches": len(c), "avg_ms": sum(c) / len(c) if c else None,
                "attn_launches": len(t), "attn_avg_ms": sum(t) / len(t) if t else None}

    def config(self):
        return {"workload": f"BASELINE cfg4: SD-2.1-base UNet (866 M params, random init) {self.STEPS}-step CFG denoise through "
                            f"StableDiffusion.generate_images, latents ({2 * self.B},4,64,64), ctx (77,1024), MMFSNet (13 blocks) on 1 "
                            "context image, DDPM scheduler (sd.py:48-50); 3x3/1x1 convs (tcgen05 implicit GEMM), GroupNorm+SiLU, GEGLU, "
                            "attention, LayerNorm, MMFS = this repo's kernels; conv_in/conv_out + Linear GEMMs = cuDNN/cuBLAS; VAE not run",
                "step_unit": f"one {self.STEPS}-step denoise of the rank-local batch of {self.B} images (2B UNet rows for CFG)",
                "images_per_step": self.B, "global_batch": self.B * self.world, "parallelism": f"dp{self.world}",
                "cuda_graph": "UNet evaluation captured once per shape and kept across generate_images calls "
                              "(StableDiffusion.enable_cuda_graphs); per call the context, mask and MMFS image-side state are "
                              "refreshed in place; scheduler steps eager; roofline kernels timed in separate eager evaluations",
                "l2": "192 MiB buffer written between timed steps"}

    def roofline(self, kernel):
        peaks = measured_peaks()
        cin, cout, side, ks = self.CONV_SHAPE
        cflops = 2.0 * (2 * self.B) * side * side * cout * cin * ks * ks
        tc = kernel["avg_ms"] * 1e-3 if kernel["avg_ms"] else None
        flops = 4.0 * (2 * self.B) * 4096 * 4096 * 320                   # self-attn at T=4096, C=320 (5 x 64)
        t = kernel["attn_avg_ms"] * 1e-3 if kernel.get("attn_avg_ms") else None
        return {"kernel": f"conv_igemm_kernel<bf16> (tcgen05 implicit GEMM), {cin}->{cout} {side}x{side} {ks}x{ks}, batch {2 * self.B}",
                "bound": "tensor", "achieved": cflops / tc / 1e12 if tc else None, "peak": peaks["bf16_tflops_sustained"],
                "unit": "TFLOP/s", "frac": cflops / tc / 1e12 / peaks["bf16_tflops_sustained"] if tc else None,
                "flops_per_launch": cflops, "avg_launch_us": tc * 1e6 if tc else None, "launches_timed": kernel["launches"],
                "traffic": None,
                "attention": {"kernel": "attn_fwd_kernel<bf16,64> (tcgen05), UNet self-attention at T=4096 (5 heads x 64)",
                              "bound": "tensor", "achieved": flops / t / 1e12 if t else None,
                              "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                              "frac": flops / t / 1e12 / peaks["bf16_tflops_sustained"] if t else None,
                              "avg_launch_us": t * 1e6 if t else None, "launches_timed": kernel.get("attn_launches")}}

    def cpu_baseline(self):
        return {"value": None, "unit": self.unit, "cores": 0, "kind": "port",
                "sample": "not timed: the UNet restatement (oracle/unet.py) at 512^2 x 50 steps x 16 rows is hours of CPU work"}


# ----------------------------------------------------------------------------------------------------------
class GenerateCfg5(Workload):
    """BASELINE cfg 5: end-to-end ``generate(mode="generate_texts")`` then ``generate(mode="generate_images")`` on an
    8-image interleaved context (inference.py:237-269 alternates the two modes per sample; batch 1 per call like
    inference.py:100-109).  Text: 30 new tokens, greedy (SURVEY.md 8d: greedy for determinism; eos suppressed so
    every step decodes the full 30).  Image: the LAST image of the context is the target (inference.py:98), 30 denoise
    steps, guidance 7.5 (mm_inference.yaml:55-56), latents returned (no VAE)."""

    name = "generate_cfg5"
    metric = "generate_texts_plus_images_samples_per_sec"
    unit = "steps/s"
    T, N_IMG, TOK_PER_IMG, NEW_TOKENS, DENOISE = 1024, 8, 64, 30, 30
    default_steps, default_warmup = 2, 2      # graph captures (decode step, UNet evaluation), then first-use allocations

    def setup(self):
        self.model = full_model()
        self.model.enable_cuda_graphs(tokenizer=True)
        self.model.enable_decode_graphs(True)                 # one CUDA graph replay per generated token
        g = torch.Generator().manual_seed(99 + self.rank)
        self.host_sets = []
        for _ in range(2):
            ids = torch.randint(3, 31999, (1, self.T), generator=g)
            ids[:, 0] = BOS_ID
            for k in range(self.N_IMG):
                s = 1 + k * 128 if k < self.N_IMG - 1 else self.T - 1 - self.TOK_PER_IMG
                ids[:, s] = SOI_ID
                ids[:, s + 1:s + 1 + self.TOK_PER_IMG] = IMG_ID
            images = torch.rand((self.N_IMG, 3, 224, 224), generator=g)
            self.host_sets.append([ids.pin_memory(), images.pin_memory(), torch.tensor([self.N_IMG]).pin_memory()])
        self.host = self.host_sets[0]
        self.dev_sets = [[t.cuda() for t in st] for st in self.host_sets]
        self.tgt = torch.tensor([self.N_IMG - 1], device="cuda")
        self.out_ids_h = torch.empty((1, self.NEW_TOKENS), dtype=torch.long).pin_memory()
        self.out_img_h = torch.empty((1, 4, 64, 64), dtype=torch.bfloat16).pin_memory()
        self._i = 0
        self._text_ms, self._image_ms = [], []
        self.reset_counters()

    def teardown(self):
        self.model.enable_decode_graphs(False)

    def extras(self, value):
        tm = sum(self._text_ms) / len(self._text_ms) if self._text_ms else None
        im = sum(self._image_ms) / len(self._image_ms) if self._image_ms else None
        return {"samples_per_s": value, "generate_texts_ms": tm, "generate_images_ms": im,
                "decode_ms_per_token": None if tm is None else tm / self.NEW_TOKENS}

    def _run(self, t):
        ids, images, nimg = t
        batch = dict(text_ids=ids, image_tensors=images, num_image_per_seq=nimg, attention_mask=None, meta=None,
                     max_num_image=self.N_IMG)
        e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        e[0].record()
        txt = self.model.generate(mode="generate_texts", **batch, num_beams=1, max_length=self.NEW_TOKENS,
                                  min_length=self.NEW_TOKENS)["text_ids"]
        e[1].record()
        img = self.model.generate(mode="generate_images", **batch, target_image_idxs=self.tgt,
                                  num_inference_steps=self.DENOISE, guidance_scale=7.5)["image"]
        e[2].record()
        self._ev = e
        return txt, img

    def _note(self):
        torch.cuda.synchronize()
        self._text_ms.append(self._ev[0].elapsed_time(self._ev[1]))
        self._image_ms.append(self._ev[1].elapsed_time(self._ev[2]))

    def step_device(self):
        self.last = self._run(self.dev_sets[self._i % 2])
        self._i += 1
        self._note()

    def step_e2e(self):
        host = self.host_sets[self._i % 2]
        self._i += 1
        txt, img = self._run([t.to("cuda", non_blocking=True) for t in host])
        self.out_ids_h.copy_(txt[:, :self.NEW_TOKENS], non_blocking=True)
        self.out_img_h.copy_(img, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        self.last = (txt, img)

    def reset_counters(self):
        super().reset_counters()
        self._text_ms, self._image_ms = [], []

    def result_checksum(self):
        return (self.last[0].sum().float() + self.last[1].float().sum()).reshape(1)

    def outputs(self):
        return {"text_ids": self.last[0], "image_latents": output_sample(self.last[1])}

    def h2d_bytes(self):
        return sum(t.numel() * t.element_size() for t in self.host)

    def d2h_bytes(self):
        return self.out_ids_h.numel() * 8 + self.out_img_h.numel() * 2

    def kernel_stats(self):
        return {"launches": 0, "avg_ms": None}

    def config(self):
        return {"workload": f"BASELINE cfg5: MMInterleaved.generate(mode='generate_texts') ({self.NEW_TOKENS} new tokens, greedy, KV "
                            f"cache) then generate(mode='generate_images') ({self.DENOISE}-step CFG denoise of the last image, latents "
                            f"out) on one {self.N_IMG}-image / {self.T}-token interleaved context per call (inference.py:237-269)",
                "step_unit": "one sample: one generate_texts call + one generate_images call (batch 1)",
                "global_batch": self.world, "seq_len": self.T, "images_per_seq": self.N_IMG, "parallelism": f"dp{self.world}",
                "cuda_graph": "visual tokenizer graph + one decode-step graph replayed per generated token (enable_decode_graphs) + "
                              "the UNet evaluation graph kept across calls",
                "l2": "192 MiB buffer written between timed steps"}

    def roofline(self, kernel):
        peaks = measured_peaks()
        tm = sum(self._text_ms) / len(self._text_ms) if self._text_ms else None
        if tm is None:
            return None
        # decode floor: every generated token re-reads the decoder weights (13.0 B params bf16) + the KV cache
        wbytes = 2.0 * (40 * (4 * 5120 * 5120 + 3 * 5120 * 13824) + 10 * (5120 * 5120 + 5120 * 688 + 1024 * 5120) + 32128 * 5120)
        kv = 2.0 * 40 * 2 * self.T * 5120
        return {"kernel": "decode step (HBM-bound: weight + KV-cache read per token)", "bound": "hbm",
                "note": "generate_texts time / new tokens, INCLUDING the prefill and the visual tokenizer (upper bound of the per-token time)",
                "achieved": (wbytes + kv) / (tm * 1e-3 / self.NEW_TOKENS) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": (wbytes + kv) / (tm * 1e-3 / self.NEW_TOKENS) / 1e9 / peaks["hbm_gbs"],
                "bytes_per_token": wbytes + kv, "traffic": None}

    def cpu_baseline(self):
        return {"value": None, "unit": self.unit, "cores": 0, "kind": "port", "sample": "not timed (see cfg3's CPU baseline)"}


WORKLOADS = {"msda_cfg3": MsdaCfg3, "interleaved_cfg3": InterleavedCfg3, "interleaved_cfg2": InterleavedCfg2,
             "sd_cfg4": SdCfg4, "generate_cfg5": GenerateCfg5}
AUTO = "interleaved_cfg3"
SECONDARY = ("interleaved_cfg2", "sd_cfg4", "generate_cfg5")     # emitted as `secondary` objects beside the main line


def make(name, rank, world, local_batch):
    if name == "auto":
        name = AUTO
    return WORKLOADS[name](rank, world, local_batch)


def run_reference_arm(args, world):
    """`bench.py --impl reference`: the reference's own CPU implementation of the path timed on the host cores with all
    threads, bounded sample per step (the reference CUDA op has no CPU implementation, ops/src/ms_deform_attn.h:38, and
    a 13 B fp32 forward does not fit a bounded CPU run: the arm times the oracle restatement of the reference layers)."""
    name = AUTO if args.workload == "auto" else args.workload
    wl = WORKLOADS[name](0, world, args.local_batch)
    threads = os.cpu_count() or 1
    if name.startswith("interleaved"):
        threads = min(threads, 64)
    torch.set_num_threads(threads)
    wl.setup_cpu_only()
    for _ in range(max(min(args.warmup, 2), 1)):
        wl.reference_step()
    t0 = time.time()
    samples = [wl.reference_step() for _ in range(args.steps)]
    dt = time.time() - t0
    value = wl.reference_value(samples)
    line = {"impl": "reference", "metric": wl.metric, "value": value, "unit": wl.unit, "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 1), "ms_per_step": dt * 1e3 / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": wl.config(),
            "cpu_baseline": {"value": value, "unit": wl.unit, "cores": threads, "kind": "port",
                             "sample": wl.reference_sample},
            "e2e": {"value": value, "unit": wl.unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    line.update(wl.extras(value))
    return line
