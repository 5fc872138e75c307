"""CPU tests: pin the oracle (oracle/msda_ref.c, oracle.msda_core_pytorch) against the golden
vectors generated from the reference's own code."""
import os

import numpy as np
import pytest
import torch

from oracle import error_metrics, make_msda_inputs, msda_core_pytorch, msda_forward_ref
from tests._golden import GOLDEN, load_msda_case, msda_case_names
from tests.golden.make_golden import CORE_MODES, CORE_MODES_CASE, golden_sample, input_digest

# fp32 accumulation-order noise between the scalar restatement and grid_sample
F32_TOL = dict(max_abs=2e-6, max_rel=2e-5)


@pytest.mark.parametrize("name", msda_case_names())
def test_c_restatement_matches_reference_golden(name):
    c = load_msda_case(name)
    out = msda_forward_ref(c["value"], c["spatial_shapes"], c["level_start_index"], c["sampling_loc"], c["attn_weight"])
    m = error_metrics(out, c["out_fp64"])
    assert m["max_abs"] < F32_TOL["max_abs"] and m["max_rel"] < F32_TOL["max_rel"], m
    out64 = msda_forward_ref(c["value"].double(), c["spatial_shapes"], c["level_start_index"],
                             c["sampling_loc"].double(), c["attn_weight"].double())
    m64 = error_metrics(out64, c["out_fp64"])
    assert m64["max_abs"] < 1e-12, m64


@pytest.mark.parametrize("name", msda_case_names())
def test_pytorch_core_restatement_matches_reference_golden(name):
    c = load_msda_case(name)
    out = msda_core_pytorch(c["value"], c["spatial_shapes"], c["sampling_loc"], c["attn_weight"])
    assert torch.equal(out, c["out_fp32"])  # same ATen ops in the same order => bit identical
    out64 = msda_core_pytorch(c["value"].double(), c["spatial_shapes"], c["sampling_loc"].double(), c["attn_weight"].double())
    assert torch.equal(out64, c["out_fp64"])


def test_index_stream_fields_are_consistent():
    v, s, st, loc, a = make_msda_inputs(2, [(8, 8), (4, 6), (3, 2)], 4, 32, 21, 4, seed=7, loc_mode="edges")
    out, idx = msda_forward_ref(v, s, st, loc, a, want_index_stream=True)
    inr, h0, w0, valid = idx[..., 0], idx[..., 1], idx[..., 2], idx[..., 3]
    H = s[:, 0].view(1, 1, 1, -1, 1).int()
    W = s[:, 1].view(1, 1, 1, -1, 1).int()
    sel = inr == 1
    assert 0.2 < sel.float().mean() < 0.9           # the generator really exercises both branches
    assert (h0[sel] >= -1).all() and (h0[sel] <= (H.expand_as(h0)[sel] - 1)).all()
    assert (w0[sel] >= -1).all() and (w0[sel] <= (W.expand_as(w0)[sel] - 1)).all()
    # every partial-validity pattern the border can produce shows up
    seen = set(valid[sel].tolist())
    assert {1, 2, 4, 8, 3, 5, 10, 12, 15} <= seen, seen
    # offsets: ptr1 = (h0*W + w0)*M*D + m*D whenever corner 1 is valid
    M, D = 4, 32
    m_idx = torch.arange(M).view(1, 1, M, 1, 1).expand_as(h0)
    c1 = sel & ((valid & 1) == 1)
    expect = (h0 * W + w0) * (M * D) + m_idx * D
    assert torch.equal(idx[..., 4][c1], expect[c1].int())
    assert (idx[..., 4:][~sel] == -1).all() and (idx[..., :4][~sel] == 0).all()


def test_empty_and_degenerate_shapes():
    v, s, st, loc, a = make_msda_inputs(1, [(1, 1)], 1, 8, 3, 1, seed=3)
    out = msda_forward_ref(v, s, st, loc, a)
    ref = msda_core_pytorch(v, s, loc, a)
    assert error_metrics(out, ref)["max_abs"] < 1e-6
    # all points out of range -> exact zeros (cu:55 zero-initialised output)
    out0 = msda_forward_ref(v, s, st, loc + 5.0, a)
    assert torch.count_nonzero(out0) == 0


def test_against_live_reference_core():
    """The reference's ms_deform_attn_core_pytorch under every location mode; its outputs (a strided sample) are
    stored in tests/golden/oracle_msda_loc_modes.npz by make_golden.make_core_modes."""
    z = np.load(os.path.join(GOLDEN, "oracle_msda_loc_modes.npz"))
    N, shapes, M, D, Lq, P = CORE_MODES_CASE
    for seed, mode in enumerate(CORE_MODES):
        v, s, st, loc, a = make_msda_inputs(N, shapes, M, D, Lq, P, seed=seed, loc_mode=mode)
        assert input_digest(v, loc, a) == str(z[f"{mode}_input_sha1"]), f"inputs of mode '{mode}' do not reproduce"
        r = torch.from_numpy(z[f"{mode}_fp64"])
        o = golden_sample(msda_forward_ref(v, s, st, loc, a))
        m = error_metrics(o, r)
        assert m["max_abs"] < F32_TOL["max_abs"], (mode, m)
        assert torch.equal(golden_sample(msda_core_pytorch(v, s, loc, a)), torch.from_numpy(z[f"{mode}_fp32"]))
