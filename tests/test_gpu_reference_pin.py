"""GPU: the B200 kernels banet_eqc_fwd / banet_eqc_bwd against what the reference's OWN native op — EquationConstruction /
EquationConstructionGrad compiled unmodified from utils.cu (oracle/Makefile, against the TensorFlow stand-in headers) — computed on a B200,
and the float64 oracle against the same recorded outputs.  The recorded outputs and timings are tests/golden/ref_eqc_cases.npz,
ref_eqc.npz and ref_op_timing.json, written by tests/golden/gen_ref_eqc_golden.py.  This pins SURVEY §8 rows a8-a10."""
import json
import os

import numpy as np
import pytest
import torch

from helpers import O, rel_fro, GOLDEN_DIR
import gen_ref_eqc_golden as GR

pytestmark = pytest.mark.gpu


def _recorded(case):
    """The reference op's outputs for one case: {name: (flat indices, values)}; fails if the regenerated inputs are not the recorded ones."""
    z = np.load(os.path.join(GOLDEN_DIR, "ref_eqc_cases.npz"))
    key = GR.case_key(*case)
    inputs = GR.case_inputs(*case)
    np.testing.assert_allclose([float(t.double().sum()) for t in inputs], z[f"{key}_input_sum"], rtol=1e-12, atol=1e-9)
    return inputs, {n: (torch.from_numpy(z[f"{key}_{n}_idx"].astype(np.int64)), torch.from_numpy(z[f"{key}_{n}"])) for n in ("AtA", "Atb", "dJ", "dG", "dd")}


def _at(t, idx):
    return t.detach().reshape(-1).cpu()[idx]


@pytest.mark.parametrize("nb,N,C,P", GR.CASES)
def test_reference_op_vs_oracle_and_b200_kernels(nb, N, C, P):
    from banet_b200 import ops
    (J, G, d, lg, rg), ref = _recorded((nb, N, C, P))
    cmp = lambda name, t: rel_fro(_at(t, ref[name][0]), ref[name][1])
    oA, ob = O.equation_construction(J.double(), G.double(), d.double())
    # the reference sums N per-pixel fp32 matrices serially in fp32 (utils.cu:181-198): ~1e-6 per element
    assert rel_fro(ref["AtA"][1], _at(oA, ref["AtA"][0])) < 2e-5 and rel_fro(ref["Atb"][1], _at(ob, ref["Atb"][0])) < 2e-5
    A, b = ops.equation_construction(J.cuda(), G.cuda(), d.cuda())
    assert cmp("AtA", A) < 2e-5 and cmp("Atb", b) < 2e-5
    oJ, oG, od = O.equation_construction_grad(J.double(), G.double(), d.double(), lg.double(), rg.double())      # the 2*A*Ghat form, utils.cu:648
    for name, t in (("dJ", oJ), ("dG", oG), ("dd", od)):
        assert rel_fro(ref[name][1], _at(t, ref[name][0])) < 2e-5, name
    dJ, dG, dd = ops.equation_construction_grad(J.cuda(), G.cuda(), d.cuda(), lg.cuda(), rg.cuda(), exact_sym=False)
    assert cmp("dJ", dJ) < 2e-5 and cmp("dG", dG) < 2e-5 and cmp("dd", dd) < 2e-5
    print(f"nb={nb} N={N} C={C} P={P}: ref vs oracle AtA {rel_fro(ref['AtA'][1], _at(oA, ref['AtA'][0])):.1e}; "
          f"b200 vs ref AtA {cmp('AtA', A):.1e} dJ {cmp('dJ', dJ):.1e}")


def test_b200_op_reproduces_reference_golden():
    """tests/golden/ref_eqc.npz holds the inputs and outputs of the compiled reference kernel; the CPU suite holds the oracle to it
    (tests/test_oracle_pinned_eqc.py), and here the B200 kernels behind the same op boundary must reproduce it."""
    z = np.load(os.path.join(GOLDEN_DIR, "ref_eqc.npz"))
    from banet_b200 import ops
    J, G, d, lg, rg = [torch.tensor(z[k]).cuda() for k in ("in_J", "in_G", "in_d", "in_left_grad", "in_right_grad")]
    A, b = ops.equation_construction(J, G, d)
    dJ, dG, dd = ops.equation_construction_grad(J, G, d, lg, rg, exact_sym=False)
    for got, key in ((A, "out_AtA"), (b, "out_Atb"), (dJ, "out_dJ"), (dG, "out_dG"), (dd, "out_dd")):
        assert rel_fro(got, z[key]) < 1e-5, key


def test_reference_op_timed_beside_the_b200_kernels():
    """The reference's own CUDA op (cuBLAS batched SGEMM chain + its serial column reduction, utils.cu:331-414 / :613-690), as recorded on a
    B200 in tests/golden/ref_op_timing.json, beside the B200 kernels behind the same op boundary timed here on the same inputs, at the
    reference's own scale (nb=2, 4096 sampled points, legacy/seq_example.py:12) and at a 160x120 level.  Also the fused layer-level build
    (never materialises J, G, d) at the same shape.  Report only (printed); the single assertion is that the replacement is not slower.
    Margin: when the record was taken, the B200 kernels timed on the same B200 were 23x (forward) and 59x (backward) faster at nb=2,
    N=4096 and 35x / 70x at nb=4, N=19200, so only a slowdown of more than 20x on the box running the test can fail it."""
    from banet_b200 import ops, synth
    rec = json.load(open(os.path.join(GOLDEN_DIR, "ref_op_timing.json")))
    print("reference op recorded on:", rec["gpu"])
    for (nb, gh, gw), row in zip(GR.TIMING_SHAPES, rec["rows"]):
        assert (row["nb"], row["N"]) == (nb, gh * gw)
        J, G, d, lg, rg = [t.cuda() for t in GR.timing_inputs(nb, gh, gw)]
        row = dict(row, b200_eqc_fwd_ms=GR.wall_ms(lambda: ops.equation_construction(J, G, d)),
                   b200_eqc_bwd_ms=GR.wall_ms(lambda: ops.equation_construction_grad(J, G, d, lg, rg)))
        del J, G, d
        C, K = 128, 128
        sc = synth.make_scene(nb=nb, H=gh, W=gw, C=C, K=K, level_ids=(3,), seed=11, device="cuda", dtype=torch.float32)
        lv = sc.levels[0]; L = ops.Level(lv.conv1, lv.conv2, lv.intr, lv.p, lv.D, lv.B, grid=lv.grid)
        row["b200_fused_build_fp32_ms"] = GR.wall_ms(lambda: ops.lm_build(L, sc.R0, sc.T0, sc.W0, precision=0))
        row["b200_fused_build_auto_ms"] = GR.wall_ms(lambda: ops.lm_build(L, sc.R0, sc.T0, sc.W0, precision=-1))
        print(row, f"reference / b200: forward {row['reference_fwd_ms'] / row['b200_eqc_fwd_ms']:.1f}x, "
                   f"backward {row['reference_bwd_ms'] / row['b200_eqc_bwd_ms']:.1f}x")
        assert row["b200_eqc_fwd_ms"] < row["reference_fwd_ms"] and row["b200_eqc_bwd_ms"] < row["reference_bwd_ms"]
