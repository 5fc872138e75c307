"""CPU tests: pin oracle/mmfs.py (restatement of MMFS.forward, mmfs.py:120-276) against the committed
outputs of the reference module."""
import glob
import os

import numpy as np
import pytest
import torch

from oracle import error_metrics
from oracle.mmfs import mmfs_forward_ref

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
NAMES = sorted(os.path.basename(p)[5:-4] for p in glob.glob(os.path.join(GOLDEN, "mmfs_*.npz")))


def load_mmfs_case(name):
    from tests.golden.make_golden import MMFS_CASES
    z = np.load(os.path.join(GOLDEN, f"mmfs_{name}.npz"))
    params = {k[len("param/"):]: torch.from_numpy(z[k]) for k in z.files if k.startswith("param/")}
    t = {k: torch.from_numpy(z[k]) for k in z.files if not k.startswith("param/")}
    c = MMFS_CASES[name]["ctor"]
    kw = dict(n_heads=c["n_heads"], n_levels=c["n_levels"], n_points=c["n_points"],
              scale_ratios=torch.tensor([s / c["base_spatial_shape"] for s in c["spatial_shapes"]]))
    return params, t, kw, MMFS_CASES[name]


@pytest.mark.parametrize("name", NAMES)
def test_mmfs_restatement_matches_reference_golden(name):
    params, t, kw, _ = load_mmfs_case(name)
    out = mmfs_forward_ref(params, t["query"], t["reference_points"], t["input_flatten"], t["spatial_shapes"],
                           t["level_start_index"], t["attention_mask"], **kw)
    m = error_metrics(out, t["out_fp32"])
    assert m["max_abs"] < 2e-6, m          # same ops, same order up to reshapes
    p64 = {k: v.double() for k, v in params.items()}
    out64 = mmfs_forward_ref(p64, t["query"].double(), t["reference_points"].double(), t["input_flatten"].double(),
                             t["spatial_shapes"], t["level_start_index"], t["attention_mask"].double(),
                             **{**kw, "scale_ratios": kw["scale_ratios"].double()})
    assert error_metrics(out64, t["out_fp64"])["max_abs"] < 1e-10


def test_mmfs_restatement_against_live_reference():
    """A second llm_tiny-shaped case with seeded weights; the reference module's output on it is stored in
    tests/golden/oracle_mmfs_seeded.npz by make_golden.make_mmfs_seeded."""
    from tests.golden.make_golden import MMFS_SEEDED, mmfs_case_inputs, mmfs_seeded_state_dict
    case = MMFS_SEEDED
    z = np.load(os.path.join(GOLDEN, "oracle_mmfs_seeded.npz"))
    template, _, _, _ = load_mmfs_case("llm_tiny")              # same constructor: parameter names and shapes
    sd = mmfs_seeded_state_dict(template)
    assert float(sum(v.double().sum() for v in sd.values())) == float(z["weight_checksum"]), "seeded weights drifted"
    query, refpts, feat, ss, starts, mask = mmfs_case_inputs(case)
    want = torch.from_numpy(z["out_fp32"])
    c = case["ctor"]
    got = mmfs_forward_ref(sd, query, refpts, feat, ss, starts, mask, n_heads=c["n_heads"],
                           n_levels=c["n_levels"], n_points=c["n_points"],
                           scale_ratios=torch.tensor([s / c["base_spatial_shape"] for s in c["spatial_shapes"]]))
    assert error_metrics(got, want)["max_abs"] < 2e-6
