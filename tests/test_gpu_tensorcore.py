"""GPU tests of the tcgen05 / TMA building blocks (SWIZZLE_128B MN-major operands, kind::tf32) against fp64 matmul."""
import pytest
import torch

from helpers import rel_fro

pytestmark = pytest.mark.gpu


def _selftest(A, R, mode, use_rna, repeat=1):
    from banet_b200 import _lib
    lib = _lib.load(); _lib.require_device()
    D = torch.full((128, 160), float("nan"), device="cuda")
    _lib.check(lib.banet_tc_selftest(A.data_ptr(), R.data_ptr(), D.data_ptr(), mode, use_rna, repeat, torch.cuda.current_stream().cuda_stream),
               "banet_tc_selftest")
    torch.cuda.synchronize()
    return D


def _tf32_exact(x):
    return (x.view(torch.int32) & -8192).view(torch.float32)          # 10-bit mantissa: exactly representable in tf32


def test_tcgen05_layout_exact_on_tf32_representable_inputs():
    g = torch.Generator().manual_seed(0)
    A = _tf32_exact(torch.randn(64, 128, generator=g)).cuda(); R = _tf32_exact(torch.randn(64, 160, generator=g)).cuda()
    D = _selftest(A, R, 0, 0)
    ref = A.double().t() @ R.double()
    assert torch.isfinite(D).all()
    assert rel_fro(D, ref) < 1e-6          # only fp32 accumulation error remains: layout + descriptors are right


def test_tcgen05_index_pattern():
    """A and R with one-hot structure: D[i,j] must pick exactly A[k,i]*R[k,j] — catches any swizzle/stride mix-up."""
    A = torch.zeros(64, 128); R = torch.zeros(64, 160)
    for k in range(64):
        A[k, (3 * k + 1) % 128] = float(k + 1); R[k, (7 * k + 2) % 160] = 1.0
    D = _selftest(A.cuda(), R.cuda(), 0, 0)
    assert torch.equal(D.cpu(), A.t() @ R)


@pytest.mark.parametrize("mode,use_rna,tol", [(0, 0, 2e-3), (0, 1, 1e-3), (1, 1, 3e-4), (1, 0, 1e-3)])
def test_tcgen05_precision_modes(mode, use_rna, tol):
    g = torch.Generator().manual_seed(1)
    A = torch.randn(64, 128, generator=g).cuda(); R = torch.randn(64, 160, generator=g).cuda()
    D = _selftest(A, R, mode, use_rna)
    err = rel_fro(D, A.double().t() @ R.double())
    print(f"mode={mode} rna={use_rna} rel-fro={err:.3e}")
    assert err < tol


def test_tcgen05_accumulator_rounding():
    """Accumulate the same (tf32-exact, positive) tile T times: the exact answer is T * D1.  Documents how the TMEM fp32
    accumulator rounds (printed).  Measured on B200: every accumulation step TRUNCATES (mean -5e-8 relative per step),
    which is why lm_build_tc keeps TMEM chains short and adds them up round-to-nearest outside the tensor core."""
    g = torch.Generator().manual_seed(3)
    A = _tf32_exact(torch.rand(64, 128, generator=g) + 0.5).cuda(); R = _tf32_exact(torch.rand(64, 160, generator=g) + 0.5).cuda()
    ref1 = A.double().t() @ R.double()
    for T in (1, 16, 256):
        D = _selftest(A, R, 0, 0, repeat=T).double()
        rel = ((D - T * ref1) / (T * ref1))
        print(f"T={T}: mean rel err {rel.mean().item():+.3e}  rms {rel.pow(2).mean().sqrt().item():.3e}  max|.| {rel.abs().max().item():.3e}")
        assert rel.abs().max().item() < 1.2e-7 * 8 * T          # at most one ulp per accumulation step (8 per tile)
        assert rel.mean().item() <= 0.0                           # biased toward zero
    Dn = _selftest(-A, R, 0, 0, repeat=256).double()
    reln = (Dn + 256 * ref1) / (256 * ref1)
    print(f"negated A, T=256: mean rel err of |D| {reln.mean().item():+.3e}  (negative => magnitude shrinks => round toward zero)")


# ------------------------------------------------------------------------------------ full tensor-core build path
from helpers import O, scene_case, oracle_level_inputs, to_cuda32


def _build_case(C, fly, n_points, seed, nb=3, H=48, W=64, grid=False):
    from banet_b200 import ops
    sc = scene_case(nb=nb, H=H, W=W, C=C, K=128, level_ids=(3,), seed=seed, n_points=n_points, dtype=torch.float32)
    lv = sc.levels[0]
    conv2 = lv.conv2[..., :C] if fly else lv.conv2
    lvl = ops.Level(to_cuda32(lv.conv1), to_cuda32(conv2), to_cuda32(lv.intr), to_cuda32(lv.p), to_cuda32(lv.D), to_cuda32(lv.B),
                    grid=lv.grid if grid else None)
    Wt = sc.W0 + 0.01 * torch.randn(sc.W0.shape, generator=torch.Generator().manual_seed(1))
    a = oracle_level_inputs(lv)
    ref = O.normal_equations_structured(a["conv1"], a["conv2"], a["fx"], a["fy"], a["ox"], a["oy"], a["p"], a["D"], a["B"],
                                        sc.R0.double(), sc.T0.double(), Wt.double())
    return ops, sc, lvl, Wt, ref


@pytest.mark.parametrize("C,fly,n_points,grid,hw", [(128, False, None, False, (48, 64)), (128, True, None, True, (48, 64)), (64, False, 1000, False, (48, 64)),
                                                    (64, True, 777, False, (48, 64)), (128, False, 100, False, (48, 64)),
                                                    (128, False, None, True, (48, 64)), (64, True, None, True, (44, 52)), (64, False, None, True, (20, 36))])
@pytest.mark.parametrize("prec", [1, 2, 3])
def test_lm_build_tensorcore_matches_oracle(C, fly, n_points, grid, hw, prec):
    ops, sc, lvl, Wt, (rH, rg, rrbar, rnv) = _build_case(C, fly, n_points, seed=40 + C + (n_points or 0), grid=grid, H=hw[0], W=hw[1])
    H, g, rbar, nvalid = ops.lm_build(lvl, to_cuda32(sc.R0), to_cuda32(sc.T0), to_cuda32(Wt), precision=prec)
    Hs, gs, rbs, nvs = ops.lm_build(lvl, to_cuda32(sc.R0), to_cuda32(sc.T0), to_cuda32(Wt), precision=0)
    assert torch.equal(nvalid.cpu().double(), rnv)
    eH, eg = rel_fro(H, rH), rel_fro(g, rg.squeeze(-1))
    print(f"C={C} fly={fly} grid={grid} N={sc.levels[0].N} prec={prec}: relH={eH:.2e} relg={eg:.2e}  (simt: {rel_fro(Hs, rH):.2e} {rel_fro(gs, rg.squeeze(-1)):.2e})")
    tol = {1: 5e-4, 2: 1e-4, 3: 2e-6}[prec]
    assert eH < tol and eg < tol
    # pose block and rbar do not go through the tensor cores: fp32-exact
    assert rel_fro(H[:, :6, :6], rH[:, :6, :6]) < 2e-5 and rel_fro(g[:, :6], rg[:, :6, 0]) < 2e-5
    assert rel_fro(rbar / sc.levels[0].N, rrbar.squeeze(1)) < 2e-5
    assert torch.equal(H, H.transpose(1, 2))


_PORTABLE_CASE = r'''
import sys, torch
sys.path[:0] = sys.argv[2:]
torch.backends.mkldnn.enabled = False
from helpers import O, scene_case, oracle_level_inputs
sc = scene_case(nb=2, H=96, W=128, C=64, K=128, level_ids=(2, 3), seed=91, dtype=torch.float32)

def oracle(dtype):
    olv = []
    for l in sc.levels:
        a = oracle_level_inputs(l, dtype)
        olv.append(O.LevelInputs(a["conv1"], a["conv2"], a["fx"], a["fy"], a["ox"], a["oy"], a["p"], a["D"], a["B"], []))
    opts = O.IterOptions(lambda_override=torch.full((2,), 0.05, dtype=dtype))
    return O.lm_solve(olv, 3, sc.R0.to(dtype), sc.T0.to(dtype), sc.W0.to(dtype), opts)

torch.save({"levels": [{k: getattr(l, k) for k in ("conv1", "conv2", "intr", "p", "D", "B")} for l in sc.levels],
            "R0": sc.R0, "T0": sc.T0, "W0": sc.W0, "oracle64": oracle(torch.float64), "oracle32": oracle(torch.float32)}, sys.argv[1])
'''


def _portable_cpu_case(tmp_dir):
    """The scene of test_lm_run_tensorcore_vs_oracle_outputs and the oracle's float64 and float32 solves of it, computed with CPU
    arithmetic that does not depend on the host: MKL in conditional-numerical-reproducibility mode, ATen's baseline kernels and oneDNN
    off (each selects instruction-set-specific float32 kernels otherwise).  Both settings are read when torch loads, hence the subprocess."""
    import os, subprocess, sys
    here = os.path.dirname(os.path.abspath(__file__))
    out = os.path.join(str(tmp_dir), "case.pt")
    env = dict(os.environ, MKL_CBWR="COMPATIBLE", ATEN_CPU_CAPABILITY="default")
    subprocess.run([sys.executable, "-c", _PORTABLE_CASE, out, here, os.path.dirname(here)], env=env, check=True)
    return torch.load(out)


def test_lm_run_tensorcore_vs_oracle_outputs(tmp_path):
    """Whole solve (2 levels x 3 iterations, fixed lambda, K=128) in every precision mode against the float64 oracle.
    Bar: the 1e-4 north-star tolerance on R, T, W — or, where the problem is too ill-conditioned for ANY fp32
    implementation, twice the error of the oracle itself run in float32 (the reference's arithmetic type).
    The case and both oracle runs come from _portable_cpu_case: with the host's own float32 CPU kernels, the scene and
    the float32 oracle's W error depend on the CPU the test runs on (8e-5 to 4.5e-4 across the ISA paths of one CPU)."""
    from banet_b200 import ops
    case = _portable_cpu_case(tmp_path)
    levels = [ops.Level(*[to_cuda32(l[k]) for k in ("conv1", "conv2", "intr", "p", "D", "B")]) for l in case["levels"]]
    oR, oT, oW = case["oracle64"]
    fR, fT, fW = case["oracle32"]
    floor = (rel_fro(fR, oR), rel_fro(fT, oT), rel_fro(fW, oW))
    print(f"oracle fp32 vs fp64 (noise floor): {floor[0]:.2e} {floor[1]:.2e} {floor[2]:.2e}")
    for prec in (0, 3, 2, 1):
        R, T, W, status = ops.lm_run(levels, 3, *[to_cuda32(case[k]) for k in ("R0", "T0", "W0")], lambda_fixed=0.05, precision=prec)
        errs = (rel_fro(R, oR), rel_fro(T, oT), rel_fro(W, oW))
        print(f"prec={prec}: rel-fro R,T,W = {errs[0]:.2e} {errs[1]:.2e} {errs[2]:.2e}")
        assert status.abs().max().item() == 0
        if prec in (0, 3):
            for e, f in zip(errs, floor):
                assert e < max(1e-4, 2.0 * f)


@pytest.mark.parametrize("fly,grid", [(False, True), (True, True), (False, False)])
@pytest.mark.parametrize("prec", [1, 2, 3])
def test_lm_build_tensorcore_long_tile_runs(prec, fly, grid):
    """Many tiles per CTA (ring wrap of the TMA stages and record buffers, several TMEM chains and two pair spans per CTA):
    240x320, 2 pairs = 2400 tiles over 148 CTAs.  Checked against the FP32 SIMT path (itself pinned to the oracle above),
    plus run-to-run bit reproducibility."""
    from banet_b200 import ops, synth
    sc = synth.make_scene(nb=2, H=240, W=320, C=128, K=128, level_ids=(3,), seed=17, device="cuda", dtype=torch.float32)
    lv = sc.levels[0]
    conv2 = lv.conv2[..., :128].contiguous() if fly else lv.conv2
    L = ops.Level(lv.conv1, conv2, lv.intr, lv.p, lv.D, lv.B, grid=lv.grid if grid else None)
    Wt = sc.W0 + 0.01 * torch.randn(sc.W0.shape, generator=torch.Generator().manual_seed(3)).cuda()
    Hs, gs, rbs, nvs = ops.lm_build(L, sc.R0, sc.T0, Wt, precision=0)
    H, g, rbar, nv = ops.lm_build(L, sc.R0, sc.T0, Wt, precision=prec)
    H2, g2, rbar2, nv2 = ops.lm_build(L, sc.R0, sc.T0, Wt, precision=prec)
    assert torch.equal(H, H2) and torch.equal(g, g2) and torch.equal(rbar, rbar2)
    assert torch.equal(nv, nvs)
    tol = {1: 5e-4, 2: 1e-4, 3: 2e-6}[prec]
    eH, eg = rel_fro(H, Hs), rel_fro(g, gs)
    print(f"prec={prec} fly={fly} grid={grid}: relH={eH:.2e} relg={eg:.2e}")
    assert eH < tol and eg < tol
    assert rel_fro(H[:, :6, :6], Hs[:, :6, :6]) < 2e-5 and rel_fro(rbar, rbs) < 2e-5


def test_cfg4_window_sparse_points_solve():
    """BASELINE.json configs[3] shape, scaled to test size: a keyframe tracked against 4 frames = 4 independent pairs (the reference
    has no joint multi-view solve, SURVEY §8d) on 4096 random sub-pixel points (seq_example.py:12), K=128, 10 LM iterations at a
    fixed lambda, through the tensor-core kernel's ragged (non-grid) path.  FP32 and TF32X3 must meet the north-star tolerance
    (or twice the float32 oracle's own error where the problem is too ill-conditioned for fp32); the faster modes are printed."""
    from banet_b200 import ops
    sc = scene_case(nb=4, H=240, W=320, C=64, K=128, level_ids=(3,), seed=404, n_points=4096, dtype=torch.float32)
    lv = sc.levels[0]
    level = [ops.Level(to_cuda32(lv.conv1), to_cuda32(lv.conv2), to_cuda32(lv.intr), to_cuda32(lv.p), to_cuda32(lv.D), to_cuda32(lv.B))]

    def oracle(dtype):
        a = oracle_level_inputs(lv, dtype)
        ol = [O.LevelInputs(a["conv1"], a["conv2"], a["fx"], a["fy"], a["ox"], a["oy"], a["p"], a["D"], a["B"], [])]
        return O.lm_solve(ol, 10, sc.R0.to(dtype), sc.T0.to(dtype), sc.W0.to(dtype), O.IterOptions(lambda_override=torch.full((4,), 0.5, dtype=dtype)))

    oR, oT, oW = oracle(torch.float64)
    fR, fT, fW = oracle(torch.float32)
    floor = (rel_fro(fR, oR), rel_fro(fT, oT), rel_fro(fW, oW))
    print(f"oracle fp32 vs fp64 (noise floor): {floor[0]:.2e} {floor[1]:.2e} {floor[2]:.2e}")
    for prec in (0, 3, 2, 1):
        R, T, W, status = ops.lm_run(level, 10, to_cuda32(sc.R0), to_cuda32(sc.T0), to_cuda32(sc.W0), lambda_fixed=0.5, precision=prec)
        errs = (rel_fro(R, oR), rel_fro(T, oT), rel_fro(W, oW))
        print(f"prec={prec}: rel-fro R,T,W = {errs[0]:.2e} {errs[1]:.2e} {errs[2]:.2e}")
        assert status.abs().max().item() == 0
        if prec in (0, 3):
            for e, f in zip(errs, floor):
                assert e < max(1e-4, 2.0 * f)


@pytest.mark.parametrize("K", [64, 32])
def test_small_basis_counts_on_the_tensor_cores(K):
    """K = 64 / 32 (BASELINE.json configs[4], the K sweep): the generation-6 kernel with KBLK = K / 32 basis blocks against the float64
    oracle, with and without the dense-grid hint, in the two- and three-pass modes (the single-pass mode is instantiated for K = 128 only, so
    AUTO resolves to TF32X2 here) and against the FP32 SIMT path.  First measured in round 2 (profiles/r02a_small_k_check.txt: relH 1.0e-7 /
    2.6e-8 / 2.4e-8 for X2 / X3 / FP32)."""
    from banet_b200 import ops, synth, _lib
    sc = synth.make_scene(nb=3, H=96, W=128, C=64, K=K, level_ids=(3,), seed=50 + K, device="cpu", dtype=torch.float32)
    lv = sc.levels[0]
    a = oracle_level_inputs(lv)
    Wt = sc.W0 + 0.01 * torch.randn(sc.W0.shape, generator=torch.Generator().manual_seed(1))
    rH, rg, _, rnv = O.normal_equations_structured(a["conv1"], a["conv2"], a["fx"], a["fy"], a["ox"], a["oy"], a["p"], a["D"], a["B"],
                                                   sc.R0.double(), sc.T0.double(), Wt.double())
    cu = lambda t: t.cuda()
    for grid in (None, lv.grid):
        L = ops.Level(cu(lv.conv1), cu(lv.conv2), cu(lv.intr), cu(lv.p), cu(lv.D), cu(lv.B), grid=grid)
        for prec, tol in ((_lib.PREC_FP32_SIMT, 2e-7), (_lib.PREC_TF32X2, 1e-6), (_lib.PREC_TF32X3, 2e-7), (_lib.PREC_AUTO, 1e-6)):
            H, g, rbar, nv = ops.lm_build(L, cu(sc.R0), cu(sc.T0), cu(Wt), precision=prec)
            eH, eg = rel_fro(H, rH), rel_fro(g, rg.squeeze(-1))
            print(f"K={K} grid={grid is not None} prec={prec}: relH {eH:.2e} relg {eg:.2e}")
            assert eH < tol and eg < tol, (K, grid is not None, prec, eH, eg)
            assert torch.equal(nv.cpu().double(), rnv)
