"""GPU parity tests of the native op (through the C ABI) against the CPU oracle.

Tolerances (stated here once):
  * sampling-point index math: BIT-EXACT (index stream compared field by field);
  * fp32 values: max-abs <= 2e-6 and max-rel <= 2e-5 against the fp32 scalar oracle (fp32
    re-association / FMA contraction only), and <= 1e-3 rel against the fp64 golden;
  * fp16 / bf16 values: every element within ONE storage ulp of the oracle's fp32 accumulator
    (a single rounding at the store, cuh:300), > 97 % of elements identical to the
    correctly rounded accumulator;
  * fp64: max-abs <= 1e-12.
"""
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import error_metrics, make_msda_inputs, msda_forward_ref  # noqa: E402
from tests._golden import load_msda_case, msda_case_names  # noqa: E402

DEV = "cuda"


def _mod():
    import mm_interleaved_b200 as m
    return m


def run_cuda(value, shapes, starts, loc, attn, dtype, strict=False):
    m = _mod()
    args = [value.to(DEV, dtype), shapes.to(DEV), starts.to(DEV), loc.to(DEV, dtype), attn.to(DEV, dtype)]
    out = m.ms_deform_attn_forward(*args, 64, strict=strict)
    torch.cuda.synchronize()
    return out


def assert_values_close(out, ref_acc, dtype):
    """out: CUDA result in dtype; ref_acc: oracle accumulator (fp32 or fp64, un-rounded)."""
    out = out.cpu()
    assert out.shape == ref_acc.shape
    assert torch.isfinite(out.float()).all()
    if dtype == torch.float64:
        assert (out - ref_acc).abs().max() <= 1e-12
        return
    if dtype == torch.float32:
        m = error_metrics(out, ref_acc)
        assert m["max_abs"] <= 2e-6 and m["max_rel"] <= 2e-5, m
        return
    ulp_rel = 2.0 ** -10 if dtype == torch.float16 else 2.0 ** -7
    rounded = ref_acc.to(dtype)
    diff = (out.double() - ref_acc.double()).abs()
    tol = ref_acc.double().abs() * ulp_rel + 1e-7
    assert (diff <= tol).all(), float((diff / tol).max())
    same = (out == rounded).float().mean().item()
    assert same > 0.97, same


CASES = [
    # N, shapes, M, D, Lq, P
    (2, [(8, 8), (4, 6), (3, 2)], 4, 32, 37, 4),                      # fast path D=32
    (1, [(32, 32), (16, 16), (8, 8)] * 2, 16, 64, 33, 8),             # LLM flavour, 2 images
    (1, [(64, 64), (32, 32), (16, 16), (8, 8)], 16, 64, 64, 8),       # SD flavour
    (2, [(16, 16)], 16, 32, 50, 4),                                   # ViT-Adapter extractor flavour
    (1, [(5, 7), (2, 3)], 3, 24, 9, 3),                               # generic path (D=24, P=3)
    (3, [(9, 5)], 2, 128, 17, 5),                                     # D=128, P not a power of two
    (1, [(4, 4)] * 48, 2, 64, 5, 2),                                  # many levels
    (2, [(7, 3), (1, 1)], 1, 64, 1, 1),                               # decode-like Lq=1, 1x1 level
]


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("mode", ["uniform", "clustered", "edges"])
@pytest.mark.parametrize("case", range(len(CASES)))
def test_values_match_oracle(case, mode, dtype):
    N, shapes, M, D, Lq, P = CASES[case]
    v, s, st, loc, a = make_msda_inputs(N, shapes, M, D, Lq, P, seed=100 + case, loc_mode=mode, dtype=dtype)
    ref = msda_forward_ref(v, s, st, loc, a)
    out = run_cuda(v, s, st, loc, a, dtype)
    assert_values_close(out, ref, dtype)


@pytest.mark.parametrize("case", [0, 4])
def test_fp64_matches_oracle(case):
    N, shapes, M, D, Lq, P = CASES[case]
    v, s, st, loc, a = make_msda_inputs(N, shapes, M, D, Lq, P, seed=7, loc_mode="clustered", dtype=torch.float64)
    ref = msda_forward_ref(v, s, st, loc, a)
    out = run_cuda(v, s, st, loc, a, torch.float64)
    assert_values_close(out, ref, torch.float64)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("mode", ["uniform", "clustered", "edges"])
def test_index_stream_bit_exact(mode, dtype):
    m = _mod()
    N, shapes, M, D, Lq, P = 2, [(32, 32), (16, 16), (8, 8), (24, 40), (3, 5)], 4, 64, 301, 8
    v, s, st, loc, a = make_msda_inputs(N, shapes, M, D, Lq, P, seed=11, loc_mode=mode, dtype=dtype)
    _, idx_ref = msda_forward_ref(v, s, st, loc, a, want_index_stream=True)
    idx = m.msda_index_stream(s.to(DEV), st.to(DEV), loc.to(DEV, dtype), M, D).cpu()
    assert idx.shape == idx_ref.shape
    assert torch.equal(idx, idx_ref), f"{(idx != idx_ref).any(-1).sum().item()} records differ"
    assert 0.05 < idx_ref[..., 0].float().mean() <= 1.0


def test_index_stream_full_mantissa_large():
    """20 M full-mantissa fp32 coordinates (SURVEY.md 8a': the vacuity trap of torch.rand)."""
    m = _mod()
    g = torch.Generator().manual_seed(5)
    shapes = torch.tensor([(8, 8), (16, 16), (24, 24), (32, 32), (64, 64)])
    from oracle import level_start_index
    st = level_start_index(shapes)
    N, Lq, M, L, P = 1, 25000, 16, 5, 10
    loc = (torch.rand((N, Lq, M, L, P, 2), generator=g, dtype=torch.float64) * 1.2 - 0.1).float()
    v = torch.zeros((1, int(shapes.prod(1).sum()), M, 8))
    a = torch.zeros((N, Lq, M, L, P))
    _, idx_ref = msda_forward_ref(v, shapes, st, loc, a, want_index_stream=True)
    idx = m.msda_index_stream(shapes.to(DEV), st.to(DEV), loc.to(DEV), M, 8).cpu()
    assert torch.equal(idx, idx_ref)


@pytest.mark.parametrize("name", msda_case_names())
def test_against_reference_golden(name):
    """Committed outputs of the reference's own ms_deform_attn_core_pytorch (fp64)."""
    c = load_msda_case(name)
    out = run_cuda(c["value"], c["spatial_shapes"], c["level_start_index"], c["sampling_loc"], c["attn_weight"], torch.float32)
    m = error_metrics(out, c["out_fp64"])
    assert m["max_rel"] <= 1e-3 and m["max_abs"] <= 5e-6, m
    out16 = run_cuda(c["value"], c["spatial_shapes"], c["level_start_index"], c["sampling_loc"], c["attn_weight"], torch.bfloat16)
    # bf16 storage of inputs AND output: compare against the oracle on the rounded inputs
    from oracle import round_to_dtype
    vb, lb, ab = (round_to_dtype(c[k], torch.bfloat16) for k in ("value", "sampling_loc", "attn_weight"))
    ref = msda_forward_ref(vb, c["spatial_shapes"], c["level_start_index"], lb, ab)
    assert_values_close(out16, ref, torch.bfloat16)


def test_edge_cases():
    m = _mod()
    v, s, st, loc, a = make_msda_inputs(2, [(6, 6), (3, 3)], 4, 64, 10, 4, seed=1)
    dv = lambda t: t.to(DEV)
    # empty batch / no queries
    out = m.ms_deform_attn_forward(dv(v[:0]), dv(s), dv(st), dv(loc[:0]), dv(a[:0]), 1)
    assert out.shape == (0, 10, 256)
    out = m.ms_deform_attn_forward(dv(v), dv(s), dv(st), dv(loc[:, :0]), dv(a[:, :0]), 1)
    assert out.shape == (2, 0, 256)
    # everything out of range -> exact zeros (reference: at::zeros output, cu:55)
    out = m.ms_deform_attn_forward(dv(v), dv(s), dv(st), dv(loc + 3.0), dv(a), 1)
    assert torch.count_nonzero(out) == 0
    # NaN locations fail the in-range predicate -> contribute nothing
    loc_nan = loc.clone(); loc_nan[0, 0] = float("nan")
    out = m.ms_deform_attn_forward(dv(v), dv(s), dv(st), dv(loc_nan), dv(a), 1)
    assert torch.count_nonzero(out[0, 0]) == 0 and torch.isfinite(out).all()
    # preconditions (cu:29-53)
    with pytest.raises(RuntimeError, match="contiguous"):
        m.ms_deform_attn_forward(dv(v).transpose(1, 2), dv(s), dv(st), dv(loc), dv(a), 1)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        m.ms_deform_attn_forward(dv(v), s, dv(st), dv(loc), dv(a), 1)
    with pytest.raises(RuntimeError, match="dtype"):
        m.ms_deform_attn_forward(dv(v), dv(s), dv(st), dv(loc).half(), dv(a), 1)
    v3 = torch.cat([v, v[:1]])
    with pytest.raises(RuntimeError, match="im2col_step"):
        m.ms_deform_attn_forward(dv(v3), dv(s), dv(st), dv(torch.cat([loc, loc[:1]])), dv(torch.cat([a, a[:1]])), 2)


def test_masked_images_skip_equals_strict():
    """Weights that are exactly zero (masked images after the MMFS softmax) may skip their
    fetches; the result must equal the strict path bit for bit on finite inputs."""
    v, s, st, loc, a = make_msda_inputs(2, [(32, 32), (16, 16), (8, 8)] * 4, 16, 64, 70, 8, seed=9, loc_mode="clustered")
    a = a.clone()
    a[:, :, :, 3:9] = 0        # images 1 and 2 masked for everyone
    a[0, :35, :, 0:3] = 0      # image 0 masked for half the queries of sample 0
    for dtype in (torch.float32, torch.bfloat16):
        o1 = run_cuda(v, s, st, loc, a, dtype, strict=False)
        o2 = run_cuda(v, s, st, loc, a, dtype, strict=True)
        assert torch.equal(o1, o2)
        from oracle import round_to_dtype
        ref = msda_forward_ref(round_to_dtype(v, dtype), s, st, round_to_dtype(loc, dtype), round_to_dtype(a, dtype))
        assert_values_close(o1, ref, dtype)


def test_tuning_variants_bit_identical():
    m = _mod()
    lib = m._lib.lib()
    v, s, st, loc, a = make_msda_inputs(2, [(32, 32), (16, 16), (8, 8)] * 2, 16, 64, 130, 8, seed=4, loc_mode="clustered")
    try:
        outs = []
        for rows_per_warp in (0, 1, 3, 16):
            for mapping in (0, 1):
                assert lib.mmfs_msda_set_tuning(rows_per_warp, mapping) == 0
                outs.append(run_cuda(v, s, st, loc, a, torch.bfloat16))
        for o in outs[1:]:
            assert torch.equal(o, outs[0])
    finally:
        lib.mmfs_msda_set_tuning(0, 0)


@pytest.mark.parametrize("case", [0, 3, 5, 7])
def test_small_row_kernel_agrees_with_row_kernel(case):
    """L*P <= 16 rows take the thread-per-output-vector kernel; a non-zero rows_per_warp forces the warp-per-row
    kernel on the same inputs.  Same index math, different fp32 summation order: |diff| <= 2e-6 + 2e-5 |ref| (fp32)."""
    m = _mod()
    lib = m._lib.lib()
    N, shapes, M, D, Lq, P = CASES[case]
    v, s, st, loc, a = make_msda_inputs(N, shapes, M, D, Lq, P, seed=20 + case, loc_mode="edges")
    small = run_cuda(v, s, st, loc, a, torch.float32)
    try:
        assert lib.mmfs_msda_set_tuning(2, 0) == 0
        rows = run_cuda(v, s, st, loc, a, torch.float32)
    finally:
        lib.mmfs_msda_set_tuning(0, 0)
    assert ((small - rows).abs() <= 2e-6 + 2e-5 * rows.abs()).all()


def test_full_size_properties_cfg3():
    """BASELINE cfg 3 layer shape (L=12, S=5376, Lq=2048, M=16, D=64, P=8), 2 sequences: size-
    independent properties instead of an element-wise oracle run."""
    shapes = [(32, 32), (16, 16), (8, 8)] * 4
    v, s, st, loc, a = make_msda_inputs(2, shapes, 16, 64, 2048, 8, seed=21, loc_mode="clustered")
    out = run_cuda(v, s, st, loc, a, torch.float32)
    # determinism (single writer per output, no atomics)
    assert torch.equal(out, run_cuda(v, s, st, loc, a, torch.float32))
    # batch independence: N=2 launch == two N=1 launches
    o0 = run_cuda(v[:1], s, st, loc[:1], a[:1], torch.float32)
    o1 = run_cuda(v[1:], s, st, loc[1:], a[1:], torch.float32)
    assert torch.equal(out, torch.cat([o0, o1]))
    # linearity in value
    g = torch.Generator().manual_seed(1)
    v2 = torch.rand(v.shape, generator=g)
    lin = run_cuda(0.5 * v + 2.0 * v2, s, st, loc, a, torch.float32)
    lin_ref = 0.5 * out + 2.0 * run_cuda(v2, s, st, loc, a, torch.float32)
    assert error_metrics(lin, lin_ref)["max_abs"] < 2e-5
    # partition of unity: value == 1, interior points -> out == sum of weights == 1
    loc_in = loc.clamp(0.2, 0.8)
    ones = run_cuda(torch.ones_like(v), s, st, loc_in, a, torch.float32)
    assert (ones - 1.0).abs().max() < 1e-5
    # spot-check 64 random query rows against the scalar oracle
    rows = torch.randperm(2048, generator=g)[:64]
    ref = msda_forward_ref(v, s, st, loc[:, rows].contiguous(), a[:, rows].contiguous())
    assert error_metrics(out.cpu()[:, rows], ref)["max_abs"] < 2e-6
    # bf16 at full size: one-ulp bound on the same rows
    from oracle import round_to_dtype
    ob = run_cuda(v, s, st, loc, a, torch.bfloat16)
    refb = msda_forward_ref(round_to_dtype(v, torch.bfloat16), s, st,
                            round_to_dtype(loc[:, rows].contiguous(), torch.bfloat16),
                            round_to_dtype(a[:, rows].contiguous(), torch.bfloat16))
    assert_values_close(ob[:, rows.to(DEV)], refb, torch.bfloat16)


def test_host_entry_point_matches_device_path():
    m = _mod()
    v, s, st, loc, a = make_msda_inputs(2, [(16, 16), (8, 8)], 8, 64, 100, 4, seed=2, dtype=torch.bfloat16)
    pin = lambda t, dt=None: (t.to(dt) if dt else t).contiguous().pin_memory()
    out_h = m.ms_deform_attn_forward_host(pin(v, torch.bfloat16), pin(s), pin(st), pin(loc, torch.bfloat16), pin(a, torch.bfloat16))
    out_d = run_cuda(v, s, st, loc, a, torch.bfloat16)
    assert torch.equal(out_h, out_d.cpu())


def test_dropin_module_and_autograd_wrapper():
    import MultiScaleDeformableAttention as MSDA
    m = _mod()
    v, s, st, loc, a = make_msda_inputs(1, [(8, 8)], 4, 32, 12, 4, seed=3)
    args = [v.to(DEV), s.to(DEV), st.to(DEV), loc.to(DEV), a.to(DEV)]
    o1 = MSDA.ms_deform_attn_forward(*args, 1)
    o2 = m.MSDeformAttnFunction.apply(*args, 1)
    assert torch.equal(o1, o2)
    # mixed dtypes (autocast-style): loc/weights fp32, value fp16 -> cast to value dtype
    o3 = m.MSDeformAttnFunction.apply(args[0].half(), args[1], args[2], args[3], args[4], 1)
    assert o3.dtype == torch.float16


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.float64])
@pytest.mark.parametrize("case", [0, 1, 2, 3, 5])
def test_against_the_reference_cuda_op(case, dtype):
    """The reference's OWN kernel (ops/src/cuda/ms_deform_im2col_cuda.cuh, compiled unmodified for sm_100a by
    oracle/build_ref.py) run on a B200 on the same inputs; its outputs (a strided sample) are stored in
    tests/golden/msda_ref_cuda_sampled.npz by make_golden.make_ref_cuda."""
    import os

    import numpy as np
    from tests.golden.make_golden import golden_sample, input_digest, ref_cuda_fwd_inputs
    m = _mod()
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "msda_ref_cuda_sampled.npz"))
    key = f"fwd{case}_{str(dtype).split('.')[-1]}"
    N, shapes, M, D, Lq, P = CASES[case]
    v, s, st, loc, a = ref_cuda_fwd_inputs(case, dtype)
    assert input_digest(v.float(), loc.float(), a.float()) == str(z[key + "_input_sha1"]), "inputs do not reproduce"
    args = [v.to(DEV, dtype), s.to(DEV), st.to(DEV), loc.to(DEV, dtype), a.to(DEV, dtype)]
    out = m.ms_deform_attn_forward(*args, 64)
    torch.cuda.synchronize()
    assert out.shape == (N, Lq, M * D)
    got, want = golden_sample(out.cpu()), torch.from_numpy(z[key])
    assert got.shape == want.shape and got.dtype == want.dtype
    if dtype == torch.float64:
        assert (got - want).abs().max() <= 1e-12
    elif dtype == torch.float32:
        assert (got - want).abs().max() <= 2e-6            # fp32 re-association only
    else:
        diff = (got.float() - want.float()).abs()
        assert (diff <= want.float().abs() * 2.0 ** -10 + 1e-7).all()      # both round one fp32 accumulator: <= 1 fp16 ulp
        assert (got == want).float().mean() > 0.97
