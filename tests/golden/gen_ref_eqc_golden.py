"""Records what the reference's OWN compiled op kernels (EquationConstruction + Grad, utils.cu, built unmodified by oracle/Makefile into
oracle/_ref/) compute, so that the GPU tests compare against the reference without needing its build.  Run on a B200 after `make -C oracle`:
    python tests/golden/gen_ref_eqc_golden.py OUTDIR
and commit the files it writes under tests/golden/:
    ref_eqc.npz          inputs and outputs of one small case (the CPU suite holds the oracle to it)
    ref_eqc_cases.npz    outputs for the CASES of tests/test_gpu_reference_pin.py (inputs are regenerated from their seeds; outputs with more
                         than SAMPLE elements are stored as a fixed seeded sample, with the sampled flat indices)
    ref_op_timing.json   the reference op's forward / backward times at two training-scale shapes, with the GPU and power limit they were taken on"""
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))

CASES = [(2, 70, 12, 22), (1, 33, 5, 6), (2, 257, 128, 134), (1, 64, 8, 38)]        # (nb, N, C, P)
SAMPLE = 2048
TIMING_SHAPES = [(2, 64, 64), (4, 120, 160)]                                         # (nb, grid h, grid w); C = K = 128, P = 134


def case_inputs(nb, N, C, P):
    """J, G, d, left_grad, right_grad of one case (CPU float32, seeded)."""
    g = torch.Generator().manual_seed(nb * 1000 + N + P)
    mk = lambda *s: torch.randn(*s, generator=g)
    return mk(nb, N, 2, P), mk(nb, N, C, 2), mk(nb, N, C, 1), mk(nb, P, P), mk(nb, P, 1)


def case_key(nb, N, C, P):
    return f"nb{nb}_N{N}_C{C}_P{P}"


def sample_index(numel, seed):
    """Flat indices of the stored sample of an output with `numel` elements (all of them when numel <= SAMPLE)."""
    if numel <= SAMPLE:
        return np.arange(numel, dtype=np.int32)
    return np.sort(torch.randperm(numel, generator=torch.Generator().manual_seed(seed))[:SAMPLE].numpy()).astype(np.int32)


def timing_inputs(nb, gh, gw):
    N, C, P = gh * gw, 128, 134
    g = torch.Generator().manual_seed(7)
    J = torch.randn(nb, N, 2, P, generator=g); G = torch.randn(nb, N, C, 2, generator=g); d = torch.randn(nb, N, C, 1, generator=g)
    return J, G, d, torch.randn(nb, P, P, generator=g), torch.randn(nb, P, 1, generator=g)


def wall_ms(fn, reps=5):
    """Median wall time of a synchronous call after one warm-up call."""
    fn(); torch.cuda.synchronize(); ts = []
    for _ in range(reps):
        t0 = time.perf_counter(); fn(); torch.cuda.synchronize(); ts.append(time.perf_counter() - t0)
    return sorted(ts)[len(ts) // 2] * 1e3


def main(out_dir):
    sys.path.insert(0, ROOT)
    from oracle import ref_lib
    os.makedirs(out_dir, exist_ok=True)
    meta = np.array([torch.cuda.get_device_name(0), torch.version.cuda])

    g = torch.Generator().manual_seed(4242)
    nb, N, C, P = 2, 96, 16, 38
    J = torch.randn(nb, N, 2, P, generator=g); G = torch.randn(nb, N, C, 2, generator=g); d = torch.randn(nb, N, C, 1, generator=g)
    lg = torch.randn(nb, P, P, generator=g); rg = torch.randn(nb, P, 1, generator=g)
    A, b = ref_lib.equation_construction(J.cuda(), G.cuda(), d.cuda())
    dJ, dG, dd = ref_lib.equation_construction_grad(J.cuda(), G.cuda(), d.cuda(), lg.cuda(), rg.cuda())
    np.savez_compressed(os.path.join(out_dir, "ref_eqc.npz"), in_J=J.numpy(), in_G=G.numpy(), in_d=d.numpy(), in_left_grad=lg.numpy(), in_right_grad=rg.numpy(),
                        out_AtA=A.cpu().numpy(), out_Atb=b.cpu().numpy(), out_dJ=dJ.cpu().numpy(), out_dG=dG.cpu().numpy(), out_dd=dd.cpu().numpy(), meta=meta)

    arrays = {"meta": meta}
    for case in CASES:
        J, G, d, lg, rg = case_inputs(*case)
        A, b = ref_lib.equation_construction(J.cuda(), G.cuda(), d.cuda())
        dJ, dG, dd = ref_lib.equation_construction_grad(J.cuda(), G.cuda(), d.cuda(), lg.cuda(), rg.cuda())
        key = case_key(*case)
        arrays[f"{key}_input_sum"] = np.array([float(t.double().sum()) for t in (J, G, d, lg, rg)])
        for i, (name, t) in enumerate((("AtA", A), ("Atb", b), ("dJ", dJ), ("dG", dG), ("dd", dd))):
            idx = sample_index(t.numel(), seed=i)
            arrays[f"{key}_{name}_idx"] = idx
            arrays[f"{key}_{name}"] = t.cpu().reshape(-1).numpy()[idx]
    np.savez_compressed(os.path.join(out_dir, "ref_eqc_cases.npz"), **arrays)

    rows = []
    for nb, gh, gw in TIMING_SHAPES:
        J, G, d, lg, rg = [t.cuda() for t in timing_inputs(nb, gh, gw)]
        rows.append({"nb": nb, "N": gh * gw, "C": 128, "P": 134,
                     "reference_fwd_ms": wall_ms(lambda: ref_lib.equation_construction(J, G, d)),
                     "reference_bwd_ms": wall_ms(lambda: ref_lib.equation_construction_grad(J, G, d, lg, rg))})
        del J, G, d
    smi = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    with open(os.path.join(out_dir, "ref_op_timing.json"), "w") as f:
        json.dump({"gpu": smi, "torch": torch.__version__, "cuda": torch.version.cuda,
                   "method": "median wall time of 5 synchronous calls after one warm-up", "rows": rows}, f, indent=1)
    print("wrote", sorted(os.listdir(out_dir)))


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit("usage: python tests/golden/gen_ref_eqc_golden.py OUTDIR")
    main(sys.argv[1])
