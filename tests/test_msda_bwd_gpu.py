"""GPU parity of the MSDA backward against (a) autograd through the CPU restatement of the reference's PyTorch core
in fp64 and (b) the reference's OWN CUDA backward (built by oracle/build_ref.py) run on a B200.
Tolerance fp32: |err| <= 1e-4 * max|ref| per tensor (atomics: summation order differs); 16-bit: 2e-2 * max|ref|."""
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda"

from oracle import make_msda_inputs, msda_core_pytorch  # noqa: E402

CASES = [(2, [(8, 8), (4, 6), (3, 2)], 4, 32, 37, 4), (1, [(32, 32), (16, 16), (8, 8)] * 2, 16, 64, 40, 8),
         (1, [(16, 16), (8, 8)], 2, 128, 19, 3)]


def autograd_truth(v, s, loc, a, go):
    v, loc, a = (t.double().requires_grad_(True) for t in (v, loc, a))
    out = msda_core_pytorch(v, s, loc, a)
    out.backward(go.double())
    return v.grad, loc.grad, a.grad


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("mode", ["uniform", "clustered"])
@pytest.mark.parametrize("case", range(len(CASES)))
def test_backward_matches_autograd_of_the_core(case, mode, dtype):
    import mm_interleaved_b200 as m
    N, shapes, M, D, Lq, P = CASES[case]
    v, s, st, loc, a = make_msda_inputs(N, shapes, M, D, Lq, P, seed=40 + case, loc_mode=mode, dtype=dtype)
    go = torch.randn((N, Lq, M * D), generator=torch.Generator().manual_seed(1)).to(dtype).float()
    want = autograd_truth(v, s, loc, a, go)
    got = m.ms_deform_attn_backward(v.to(DEV, dtype), s.to(DEV), st.to(DEV), loc.to(DEV, dtype), a.to(DEV, dtype),
                                    go.to(DEV, dtype), 64)
    tol = 1e-4 if dtype == torch.float32 else 2e-2
    for g, w, name in zip(got, want, ("grad_value", "grad_loc", "grad_attn")):
        assert g.dtype == dtype and g.shape == w.shape
        err = (g.double().cpu() - w).abs().max()
        assert err <= tol * w.abs().max() + 1e-7, (name, err.item(), w.abs().max().item())


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
def test_backward_matches_the_reference_cuda_op(dtype):
    """Its gradients (a strided sample of each, with the max |gradient| of the whole tensor) are stored in
    tests/golden/msda_ref_cuda_sampled.npz by make_golden.make_ref_cuda."""
    import os

    import numpy as np
    from tests.golden.make_golden import golden_sample, input_digest, ref_cuda_bwd_inputs
    import mm_interleaved_b200 as m
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "msda_ref_cuda_sampled.npz"))
    key = f"bwd_{str(dtype).split('.')[-1]}"
    v, s, st, loc, a, go = ref_cuda_bwd_inputs(dtype)
    assert input_digest(v.float(), loc.float(), a.float()) == str(z[key + "_input_sha1"]), "inputs do not reproduce"
    args = [v.to(DEV, dtype), s.to(DEV), st.to(DEV), loc.to(DEV, dtype), a.to(DEV, dtype), go.to(DEV)]
    got = m.ms_deform_attn_backward(*args, 64)
    tol = 1e-4 if dtype == torch.float32 else 2e-2
    for g, name in zip(got, ("grad_value", "grad_loc", "grad_attn")):
        w, w_max = torch.from_numpy(z[f"{key}_{name}"]), float(z[f"{key}_{name}_absmax"])
        assert (golden_sample(g.cpu()).float() - w.float()).abs().max() <= tol * w_max + 1e-7, name


def test_deterministic_backward_is_bit_reproducible_and_matches_the_float_atomic_path():
    """Heavily colliding taps (clustered locations, many queries per pixel): the default path (64-bit fixed-point integer
    atomics) gives bit-identical grad_value on repeated runs and agrees with the float-atomic path to fp32 summation noise."""
    import mm_interleaved_b200 as m
    N, shapes, M, D, Lq, P = 2, [(16, 16), (8, 8), (4, 4)], 8, 64, 3000, 8
    v, s, st, loc, a = make_msda_inputs(N, shapes, M, D, Lq, P, seed=9, loc_mode="clustered")
    go = torch.randn((N, Lq, M * D), generator=torch.Generator().manual_seed(3)) * 3.7
    args = [v.to(DEV), s.to(DEV), st.to(DEV), loc.to(DEV), a.to(DEV), go.to(DEV)]
    runs = [m.ms_deform_attn_backward(*args, 64) for _ in range(3)]
    for r in runs[1:]:
        for x, y in zip(runs[0], r):
            assert torch.equal(x, y)
    fast = m.ms_deform_attn_backward(*args, 64, deterministic=False)
    for x, y in zip(runs[0], fast):
        assert float((x - y).abs().max()) <= 1e-5 * float(y.abs().max()) + 1e-7
    # an all-zero incoming gradient (scale derived from max|grad_out| = 0) must not produce NaN / inf
    z = m.ms_deform_attn_backward(*args[:5], torch.zeros_like(args[5]), 64)
    assert all(bool(torch.isfinite(t).all()) and float(t.abs().max()) == 0.0 for t in z)


def test_autograd_function_round_trip():
    import mm_interleaved_b200 as m
    N, shapes, M, D, Lq, P = CASES[0]
    v, s, st, loc, a = make_msda_inputs(N, shapes, M, D, Lq, P, seed=5)
    vd, ld, ad = (t.to(DEV).requires_grad_(True) for t in (v, loc, a))
    out = m.MSDeformAttnFunction.apply(vd, s.to(DEV), st.to(DEV), ld, ad, 1)
    out.square().sum().backward()
    assert vd.grad is not None and ld.grad is not None and ad.grad is not None
    assert torch.isfinite(vd.grad).all() and vd.grad.abs().sum() > 0
