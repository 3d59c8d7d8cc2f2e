#!/usr/bin/env python
"""bench.py — LM iterations/sec of the BA layer's inner loop (BASELINE.json metric) on N B200s.

A "step" is one whole coarse-to-fine solve of BASELINE config 2 on every rank's shard:
nb=32 frame-pairs per GPU, dense levels 80x60 -> 640x480 (ΣN = 408 000 points/pair), C=128 feature
channels, K=128 depth bases, 5 LM iterations per level (20 iterations), lambda-MLP in the loop.
Frame-pairs are independent, so ranks hold disjoint shards (weak scaling) and the only collective is
one all-gather of the solved (R,T,W) at the end of each step (SURVEY.md §8e).

value      pair-iterations/s  = (total pairs) * 20 / t_step      inputs resident in HBM
e2e        the same through the public API with HOST buffers: pinned host -> device copies of every
           level tensor + the solve + device -> host read of (R,T,W), all inside the timed region
roofline   dominant kernel lm_build_kernel: algorithmic bytes 4*N*(2C+K+4)+4*(P^2+P+C) per pair
           (SURVEY.md §8d) / its CUDA-event duration, against MEASURED_PEAKS.json hbm_gbs
cpu_baseline / --impl reference
           the reference cannot execute here (TF-1.x / python2 / TF headers absent), so the reference arm is
           the oracle's reference-faithful materialised restatement (J,G,d tensors + batched matmul chain +
           LU solve, torch-CPU fp32, all host threads) on a bounded sample of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch

METRIC = "LM iters/sec (frame-pair LM iterations, 640x480x4-scale, K=128)"
UNIT = "pair-iters/s"
LEVEL_IDS = (0, 1, 2, 3)
H_FULL, W_FULL = 480, 640


DTYPE_NAME = {"auto": "tf32 level-wise (tcgen05 kind::tf32 x3 below 65536 points/pair, x1 above; f32 accumulate; everything else f32)",
              "levelwise": "tf32 level-wise (tcgen05 kind::tf32 x3 below 65536 points/pair, x1 above; f32 accumulate; everything else f32)",
              "fp32": "f32", "tf32x1": "tf32x1 (f32 accumulate)", "tf32x2": "tf32x2 split-A (f32 accumulate)", "tf32x3": "tf32x3 split-A/R (f32-grade)"}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg2", choices=["cfg2", "cfg4", "cfg5"],
                    help="BASELINE.json configs: cfg2 (default; the metric's workload, also cfg3 under torchrun), cfg4 = 5-frame window as 4 pairs, dense + "
                         "sparse 4096-point variants, 10 iterations per level; cfg5 = K sweep {32,64,128,256} at 640x480, nb=64, tensor cores vs fp32 SIMT")
    ap.add_argument("--nb", type=int, default=32, help="frame-pairs per GPU")
    ap.add_argument("--channels", type=int, default=128)
    ap.add_argument("--bases", type=int, default=128)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--e2e-chunks", type=int, default=8, help="pair chunks of the host pipeline (copy of chunk k+1 overlaps the solve of chunk k)")
    ap.add_argument("--layout", default="concat", choices=["concat", "f2"],
                    help="conv2 in HBM: 'concat' = [F2|gx|gy] (3C, the reference's BundleIteration boundary), 'f2' = F2 only, gradients on the fly")
    ap.add_argument("--no-precision-check", action="store_true")
    ap.add_argument("--tc-generation", type=int, default=0, choices=[0, 6, 7], help="diagnostic: banet_set_tuning(tc_generation) (0 = library default)")
    ap.add_argument("--motion", default="default", choices=["default", "large"],
                    help="planted relative motion of the synthetic pairs: default 1 deg / 2 cm (SURVEY.md section 8d), large 4 deg / 8 cm (less tap locality, fewer in-bounds points)")
    ap.add_argument("--e2e-boundary", default="resize", choices=["resize", "features", "concat"],
                    help="host buffers of the e2e leg: 'resize' = the reference's BundleResize boundary (bundlenet.py:332-399): the image batch's feature "
                         "pyramid, half-resolution basis / depth and intrinsics in; conv1, conv2, p, D, B derived on the device (ResizeHostSolver); "
                         "'features' = per-level tensors with F2 only ([F2|gx|gy] derived on the device); 'concat' = per-level tensors incl. the 3C tensor")
    ap.add_argument("--precision", default="auto", choices=["auto", "fp32", "tf32x1", "tf32x2", "tf32x3", "levelwise"],
                    help="contraction path of the build kernel: auto = tensor cores (tcgen05 tf32 split-A) when K=128, else fp32 SIMT")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned (R, T, W, status) to DIR/<name>.npy as float32 "
                         "(inputs are seeded, so two builds run with the same arguments can be compared output for output)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and (args.impl != "ours" or args.config != "cfg2"):
        ap.error("--dump-outputs applies to the cfg2 solve of --impl ours")
    return args


def dump_outputs(out_dir, out, status):
    """The arrays a caller of the timed step receives, as float32 .npy files (status codes are small integers: exact in float32)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    R, T, W = out
    for name, t in (("R", R), ("T", T), ("W", W), ("status", status)):
        if t is not None:
            np.save(os.path.join(out_dir, f"{name}.npy"), t.detach().float().cpu().numpy())


def algorithmic_bytes_per_pair_iter(N, C, K):
    """SURVEY.md §8d: dense level, conv1 + each F2 texel once + B + ray/depth + outputs."""
    P = 6 + K
    return 4 * N * (2 * C + K + 4) + 4 * (P * P + P + C)


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, index=0):
        self.index = index; self.lines = []; self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True); self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for nm, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------- reference arm
def usable_cores():
    """Threads this process may actually run on (cgroup / affinity aware; os.cpu_count() counts the whole host)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:                                           # cgroup v2 CPU quota, if any
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(int(quota) / int(period))))
    except Exception:
        pass
    return max(1, n)


def cpu_reference_iteration(O, lv, mlp, R, T, W, chunk):
    """One reference-faithful BundleIteration of ONE pair on the CPU, in point chunks so that a full 640x480 level fits in memory:
    per chunk the reference's materialised tensors J [1,n,2,P], G [1,n,C,2], d [1,n,C,1] and the native op's product chain
    (oracle.equation_construction == utils.cu:331-414), summed over chunks; then damping, LU solve and update (bundlenet.py:264-276)."""
    fx, fy, ox, oy = lv.intr_tiled()
    N = lv.N
    AtA = Atb = None
    rsum = 0
    for a in range(0, N, chunk):
        b = min(N, a + chunk)
        _, _, _, aux = O.bundle_iteration(lv.conv1[:, a:b], lv.conv2, fx[:, a:b], fy[:, a:b], ox[:, a:b], oy[:, a:b], lv.p[:, :, a:b],
                                          lv.D[:, a:b], lv.B[:, a:b], R, T, W, mlp, O.IterOptions(lambda_override=torch.ones(1)), return_aux=True)
        AtA = aux["AtA"] if AtA is None else AtA + aux["AtA"]
        Atb = aux["Atb"] if Atb is None else Atb + aux["Atb"]
        rsum = rsum + aux["rbar"] * float(b - a)
    avg = rsum / float(N)
    lam = 1000.0 * torch.pow(torch.linalg.norm(avg, dim=-1, keepdim=True), 2.0 + O.lambda_mlp(avg, mlp))
    diag = torch.diagonal(AtA, dim1=-2, dim2=-1)
    dvec = torch.cat([diag[:, :-1] + 1e-5, torch.zeros(1, 1)], dim=-1)
    sol = torch.linalg.solve(AtA + torch.diag_embed(dvec * lam.squeeze(-1)), Atb)
    return O._update(sol[:, :6, :], R, T, O.IterOptions())


def cpu_reference_sample(C, K, reps, seed=1234, level_id=3, chunk=38400):
    """Times the oracle's reference-faithful BundleIteration (J, G, d tensors + the op's product chain + LU, torch-CPU fp32, all usable
    host threads) on ONE WHOLE pair at the finest level (640x480, N = 307 200; chunked over points, nothing extrapolated within the
    level).  Returns (seconds per pair-iteration per rep, N, threads)."""
    from oracle import ba_oracle as O
    from banet_b200 import synth
    cores = usable_cores()
    torch.set_num_threads(cores)
    sc = synth.make_scene(nb=1, H=H_FULL, W=W_FULL, C=C, K=K, level_ids=(level_id,), seed=seed, dtype=torch.float32, device="cpu")
    lv = sc.levels[0]
    mlp = O.init_lambda_mlp(C, dtype=torch.float32)
    times = []
    with torch.no_grad():
        for i in range(reps + 1):
            t0 = time.perf_counter()
            cpu_reference_iteration(O, lv, mlp, sc.R0, sc.T0, sc.W0, chunk)
            times.append(time.perf_counter() - t0)
    return times[1:], lv.N, cores        # first call is a warm-up


def pixels_per_pair_iter():
    """A pair-iteration of the 4-level workload touches ΣN/4 points on average."""
    tot = sum((H_FULL // 2 ** (3 - l)) * (W_FULL // 2 ** (3 - l)) for l in LEVEL_IDS)
    return tot / len(LEVEL_IDS)


def cpu_stats(times, n_sample, cores):
    ts = sorted(times)
    med = ts[len(ts) // 2]
    scale = n_sample / pixels_per_pair_iter()          # a mean pair-iteration of the 4-level workload touches ΣN/4 points (per-point cost is level independent)
    return {"value": scale / med, "unit": UNIT, "cores": cores, "kind": "port",
            "min_med_max_s": [ts[0], med, ts[-1]], "reps": len(ts),
            "sample": (f"oracle's reference-faithful BundleIteration (materialised J/G/d per point chunk + the op's product chain + LU), ONE whole pair "
                       f"at 640x480 (N={n_sample}), fp32, {cores} threads (affinity/cgroup aware), {len(ts)} timed reps after 1 warm-up; value = "
                       f"N/(ΣN/4) / median: a pair-iteration of the 4-level workload touches ΣN/4 points on average")}, med


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    reps = args.steps                                  # a rep is one whole 640x480 pair-iteration (seconds each)
    times, n_sample, cores = cpu_reference_sample(args.channels, args.bases, reps)
    cb, med = cpu_stats(times, n_sample, cores)
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": len(times),
            "warmup": 1, "ms_per_step": med * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(args), "reference_arm": "oracle port (the TF-1.x reference cannot execute here; its code is pinned to the "
                                                                         "oracle through tests/test_oracle_pinned.py)"},
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def workload_name(args):
    return (f"cfg2: nb={args.nb}/GPU frame-pairs, dense levels 80x60..640x480, C={args.channels}, K={args.bases}, "
            f"{args.iters} LM iters/level, lambda-MLP")


# ----------------------------------------------------------------------------------------------- our arm
def _time_ms(fn, reps, warm=2):
    for _ in range(warm):
        fn()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(); e0.record()
    for _ in range(reps):
        fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def run_cfg4(args):
    """BASELINE configs[3]: one keyframe + 4 frames at 640x480, K=128, 10 LM iterations per level, as nb=4 independent pairs (the reference has no
    joint multi-view solve, SURVEY.md §8d): the dense 4-level variant and the sparse N=4096 variant of legacy/seq_example.py:12 (3C layout, ragged)."""
    from banet_b200 import ops, synth, _lib
    _lib.require_device()
    dev = torch.device("cuda", 0)
    C, K, nb, iters = args.channels, 128, 4, 10
    peak, peak_kind = measured_peaks()
    out = []
    for variant, npts in (("dense", None), ("sparse4096", 4096), ("dense_joint_window", None)):
        joint = variant == "dense_joint_window"          # the 4 pairs share D, B and ONE W: 6*4 + K unknowns, one solve (an extension, SURVEY.md section 8f-4)
        sc = synth.make_scene(nb=nb, H=H_FULL, W=W_FULL, C=C, K=K, level_ids=LEVEL_IDS, seed=1234 + 4, device=dev, dtype=torch.float32, n_points=npts,
                              shared_depth=joint)
        lay_f2 = npts is None
        levels = [ops.Level(l.conv1, l.conv2[..., :C].contiguous() if lay_f2 else l.conv2, l.intr, l.p, l.D, l.B, grid=l.grid) for l in sc.levels]
        g = torch.Generator().manual_seed(7)
        dims = [C, 2 * C, 4 * C, 2 * C, C, 1]
        packed = [ops.pack_mlp([(torch.randn(dims[i], dims[i + 1], generator=g) * (2.0 / dims[i]) ** 0.5, torch.zeros(dims[i + 1])) for i in range(5)]).to(dev) for _ in LEVEL_IDS]
        ws = torch.empty(ops.lm_run_workspace_bytes(levels, _lib.PREC_AUTO), dtype=torch.uint8, device=dev)
        if joint:
            ms = _time_ms(lambda: ops.lm_window_run(levels, iters, sc.R0, sc.T0, sc.W0[0], mlp_packed=packed, l2_regularizer_base=1000.0), args.steps)
            graph, ms_graph = None, None
        else:
            ms = _time_ms(lambda: ops.lm_run(levels, iters, sc.R0, sc.T0, sc.W0, mlp_packed=packed, l2_regularizer_base=1000.0, workspace=ws), args.steps)
            graph = ops.LMRunGraph(levels, iters, mlp_packed=packed, l2_regularizer_base=1000.0)       # the same call captured once into a CUDA graph
            ms_graph = _time_ms(lambda: graph.solve(sc.R0, sc.T0, sc.W0), args.steps)
        N_tot = sum(l.N for l in sc.levels)
        # sparse points: no texel reuse, every point reads its own 4 taps of the 3C map
        by = nb * iters * sum((4 * l.N * (2 * C + K + 4) if npts is None else 4 * l.N * (C + 12 * C + K + 4)) + 4 * ((6 + K) ** 2 + 6 + K + C) for l in sc.levels)
        out.append({"variant": variant, "points_per_pair_sum_levels": N_tot, "ms_per_solve": ms, "pair_iters_per_s": nb * len(levels) * iters / (ms * 1e-3),
                    "algorithmic_gbs": by / (ms * 1e-3) / 1e9, "frac_of_hbm_peak": by / (ms * 1e-3) / 1e9 / peak,
                    "launches_per_solve": 1 + len(levels) * iters * (6 if joint else 3), "ms_per_solve_cuda_graph": ms_graph,
                    "pair_iters_per_s_cuda_graph": None if ms_graph is None else nb * len(levels) * iters / (ms_graph * 1e-3)})
        del sc, levels, graph
        torch.cuda.empty_cache()
    print(json.dumps({"metric": METRIC, "unit": UNIT, "value": out[0]["pair_iters_per_s"], "n_gpus": 1, "steps": args.steps, "higher_is_better": True, "data": "synthetic",
                      "config": {"workload": "cfg4: keyframe + 4 frames as nb=4 pairs, 640x480 4-level pyramid, K=128, 10 LM iters/level; dense (F2-only layout) "
                                             "and sparse N=4096 random sub-pixel points per level ([F2|gx|gy] layout, ragged tiles)", "precision": "auto"},
                      "variants": out, "roofline": {"bound": "hbm (dense) / launch+latency (sparse)", "peak": peak, "peak_kind": peak_kind, "unit": "GB/s"}}))


def run_cfg5(args):
    """BASELINE configs[4]: depth-basis sweep K in {32,64,128,256} at 640x480 (one level), nb=64, 5 LM iterations: H_dd on tensor cores
    (tcgen05 kind::tf32, AUTO policy) vs the fp32 SIMT register-tiled path."""
    from banet_b200 import ops, synth, _lib
    _lib.require_device()
    dev = torch.device("cuda", 0)
    C, nb, iters = args.channels, args.nb if args.nb != 32 else 64, 5
    peak, peak_kind = measured_peaks()
    sc = synth.make_scene(nb=nb, H=H_FULL, W=W_FULL, C=C, K=256, level_ids=(3,), seed=1234 + 5, device=dev, dtype=torch.float32)
    l = sc.levels[0]
    f2 = l.conv2[..., :C].contiguous()
    l.conv2 = None
    torch.cuda.empty_cache()
    sweep = []
    for K in (32, 64, 128, 256):
        B = l.B[..., :K].contiguous(); W0 = sc.W0[:, :K].contiguous()
        lv = [ops.Level(l.conv1, f2, l.intr, l.p, l.D, B, grid=l.grid)]
        row = {"K": K}
        for name, prec in (("tensor_core", _lib.PREC_AUTO), ("fp32_simt", _lib.PREC_FP32_SIMT)):
            if name == "tensor_core" and K == 256:
                row[name] = None                   # K = 256 runs on the SIMT path only (no tensor-core instantiation: 2 x 272 TMEM columns > 512)
                continue
            reps = args.steps
            ms_b = _time_ms(lambda: ops.lm_build(lv[0], sc.R0, sc.T0, W0, precision=prec), reps, warm=1)
            ms_s = _time_ms(lambda: ops.lm_run(lv, iters, sc.R0, sc.T0, W0, lambda_fixed=0.05, precision=prec), reps, warm=1)
            by = nb * algorithmic_bytes_per_pair_iter(l.N, C, K)
            row[name] = {"build_ms": ms_b, "solve_ms_5_iters": ms_s, "pair_iters_per_s": nb * iters / (ms_s * 1e-3), "build_gbs": by / (ms_b * 1e-3) / 1e9,
                         "build_frac_of_hbm_peak": by / (ms_b * 1e-3) / 1e9 / peak, "build_tflops": nb * 2.0 * l.N * K * (K + 7) / (ms_b * 1e-3) / 1e12}
        sweep.append(row)
        del B, lv
        torch.cuda.empty_cache()
    best = max(r["tensor_core"]["pair_iters_per_s"] for r in sweep if r["K"] == 128 and r["tensor_core"])
    print(json.dumps({"metric": METRIC, "unit": UNIT, "value": best, "n_gpus": 1, "steps": args.steps, "higher_is_better": True, "data": "synthetic",
                      "config": {"workload": f"cfg5: K sweep at 640x480 (one dense level), nb={nb}, C={C}, 5 LM iters, fixed lambda; F2-only layout", "precision": "auto vs fp32"},
                      "sweep": sweep, "roofline": {"bound": "hbm", "peak": peak, "peak_kind": peak_kind, "unit": "GB/s",
                                                   "alg_bytes_per_pair_iter": "4*N*(2C+K+4) + 4*(P^2+P+C)", "tensor_flops_per_pair_iter": "2*N*K*(K+7)"}}))


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
        return
    if args.config == "cfg4":
        return run_cfg4(args)
    if args.config == "cfg5":
        return run_cfg5(args)

    from banet_b200 import ops, synth, _lib
    from banet_b200 import dist as bdist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    _lib.require_device()
    if world > 1:
        import torch.distributed as td
        td.init_process_group("nccl", device_id=dev)

    C, K, nb, iters = args.channels, args.bases, args.nb, args.iters
    if args.tc_generation:
        _lib.set_tuning(tc_generation=args.tc_generation)
    motion = dict(rot_deg=4.0, trans_m=0.08, start_trans_noise_m=0.02) if args.motion == "large" else {}
    sc = synth.make_scene(nb=nb, H=H_FULL, W=W_FULL, C=C, K=K, level_ids=LEVEL_IDS, seed=1234 + 2 + 1000 * rank,
                          device=dev, dtype=torch.float32, **motion)
    if args.layout == "f2":            # keep only the feature third of conv2 (the gradients are recomputed on the fly by the kernel)
        for l in sc.levels:
            l.conv2 = l.conv2[..., :C].contiguous()
    levels = [ops.Level(l.conv1, l.conv2, l.intr, l.p, l.D, l.B, grid=l.grid) for l in sc.levels]
    PREC = {"auto": _lib.PREC_AUTO, "fp32": _lib.PREC_FP32_SIMT, "tf32x1": _lib.PREC_TF32X1, "tf32x2": _lib.PREC_TF32X2,
            "tf32x3": _lib.PREC_TF32X3, "levelwise": _lib.PREC_TF32_LEVELWISE}[args.precision]
    g = torch.Generator().manual_seed(7)
    dims = [C, 2 * C, 4 * C, 2 * C, C, 1]
    packed = []
    for _ in LEVEL_IDS:       # he-normal lambda-MLP, seed 7 (reference bundlenet.py:105)
        params = [(torch.randn(dims[i], dims[i + 1], generator=g) * (2.0 / dims[i]) ** 0.5, torch.zeros(dims[i + 1])) for i in range(5)]
        packed.append(ops.pack_mlp(params).to(dev))
    ws = torch.empty(ops.lm_run_workspace_bytes(levels, PREC), dtype=torch.uint8, device=dev)
    n_levels, total_iters = len(levels), len(levels) * iters

    def step():
        R, T, W, status = ops.lm_run(levels, iters, sc.R0, sc.T0, sc.W0, mlp_packed=packed, l2_regularizer_base=1000.0, workspace=ws,
                                     precision=PREC)
        if world > 1:
            return bdist.all_gather_solution(R, T, W), status
        return (R, T, W), status

    def barrier():
        if world > 1:
            td.barrier(device_ids=[local])
        torch.cuda.synchronize()

    for _ in range(max(3, args.warmup)):
        out, status = step()
    barrier()
    assert int(status.abs().max()) == 0, "solver reported a non-SPD / non-finite system"

    # ---- accuracy of the timed precision mode on THIS workload: outputs against the FP32 SIMT path (which tests/test_gpu_default_precision.py
    #      and tests/test_gpu_parity.py hold to the float64 oracle; the oracle itself does not fit a 32-pair 640x480 batch) -----------------
    precision_check = None
    nvalid_frac = None
    if rank == 0 and not args.no_precision_check:
        rf = lambda a, b: float(((a - b).norm() / b.norm()).item())
        fin = sc.levels[-1]
        _, _, _, nv = ops.lm_build(levels[-1], sc.R0, sc.T0, sc.W0, precision=PREC)
        nvalid_frac = float(nv.mean().item()) / fin.N
        if PREC != _lib.PREC_FP32_SIMT:
            R1, T1, W1, _ = ops.lm_run(levels, iters, sc.R0, sc.T0, sc.W0, mlp_packed=packed, l2_regularizer_base=1000.0, precision=PREC)
            R0_, T0_, W0_, _ = ops.lm_run(levels, iters, sc.R0, sc.T0, sc.W0, mlp_packed=packed, l2_regularizer_base=1000.0,
                                         precision=_lib.PREC_FP32_SIMT)
            d1 = ops.depth_compose(fin.D.reshape(nb, -1), fin.B, W1); d0 = ops.depth_compose(fin.D.reshape(nb, -1), fin.B, W0_)
            errs = {"R": rf(R1, R0_), "T": rf(T1, T0_), "depth": rf(d1, d0), "W": rf(W1, W0_)}
            precision_check = {"vs": "fp32_simt path (oracle-asserted in tests/), same inputs, all levels x iterations", "rel_fro": errs, "tolerance": 1e-4,
                               "ok": max(errs.values()) < 1e-4,
                               "note": "north-star tolerance 1e-4 on the pose / depth outputs; W (depth-basis coefficients) is held to it as well"}
            del d1, d0, R1, T1, W1, R0_, T0_, W0_
    barrier()

    sampler = ClockSampler(local); sampler.start()
    ev0 = torch.cuda.Event(enable_timing=True); ev1 = torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(args.steps):
        out, status = step()
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop()
    if world > 1:
        tms = torch.tensor([ms], device=dev, dtype=torch.float64)
        td.all_reduce(tms, op=td.ReduceOp.MAX)
        ms = float(tms.item())
    ms_per_step = ms / args.steps
    value = world * nb * total_iters / (ms_per_step * 1e-3)
    if rank == 0 and args.dump_outputs is not None:
        dump_outputs(args.dump_outputs, out, status)

    # ---- roofline of the dominant kernel (lm_build_kernel), per level, CUDA events on the launch stream ----
    peak, peak_kind = measured_peaks()
    per_level = []
    for lv, sl in zip(levels, sc.levels):
        for _ in range(2):
            ops.lm_build(lv, sc.R0, sc.T0, sc.W0, precision=PREC)
        reps = 5
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); e0.record()
        for _ in range(reps):
            ops.lm_build(lv, sc.R0, sc.T0, sc.W0, precision=PREC)
        e1.record(); torch.cuda.synchronize()
        t = e0.elapsed_time(e1) / reps * 1e-3
        by = nb * algorithmic_bytes_per_pair_iter(sl.N, C, K)
        by3c = by + nb * 4 * sl.N * 2 * C          # conv2 read as the reference lays it out: [F2|gx|gy] = 3C channels per texel
        per_level.append({"level": f"{sl.w}x{sl.h}", "ms": t * 1e3, "alg_bytes": by, "gbs": by / t / 1e9, "gbs_3c_layout": by3c / t / 1e9})
    top = per_level[-1]
    # DRAM traffic of the dominant kernel per launch: from the committed ncu capture of THIS kernel / layout (profiles/lm_build_traffic.json,
    # stamped with the commit and configuration it was taken on); null when the capture is of another kernel or layout
    kname = "lm_build_kernel" if PREC == _lib.PREC_FP32_SIMT else "lm_build_tc6_kernel"
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "lm_build_traffic.json")
    if os.path.exists(tpath):
        try:
            tj = json.load(open(tpath))
            if tj.get("kernel") == kname and tj.get("layout") == args.layout and tj.get("nb") == nb:
                traffic = tj.get("dram_bytes_per_launch")
                traffic_src = {k: tj.get(k) for k in ("commit", "source", "precision")}
        except Exception:
            traffic = None
    roofline = {"bound": "hbm", "kernel": f"{kname} (+lm_reduce_kernel) @640x480", "achieved": top["gbs"], "peak": peak,
                "peak_kind": peak_kind, "unit": "GB/s", "frac": top["gbs"] / peak, "frac_3c_layout": top["gbs_3c_layout"] / peak,
                "traffic": traffic, "traffic_source": traffic_src, "per_level": per_level,
                "all_levels_gbs": sum(p["alg_bytes"] for p in per_level) / sum(p["ms"] * 1e-3 for p in per_level) / 1e9}

    # ---- e2e: host buffers -> device -> solve -> host, through the public API -------------------------------
    e2e = None
    if not args.no_e2e:
        try:
            from banet_b200.host_pipeline import numa_local_to
            with numa_local_to(dev) as numa:       # this rank's pinned host buffers next to its GPU's PCIe root (matters at N > 1 on a two-socket host)
                e2e = run_e2e(args, sc, levels, packed, ws, world, local, dev, total_iters, PREC)
            e2e["host_buffers_numa"] = numa.info
        except Exception as ex:      # e.g. not enough pinnable host memory: report, do not fake
            e2e = {"value": None, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "error": str(ex)[:200]}

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        times, n_sample, cores = cpu_reference_sample(C, K, 5)
        cpu_baseline, _ = cpu_stats(times, n_sample, cores)

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": DTYPE_NAME[args.precision],
                "data": "synthetic",
                "config": {"workload": workload_name(args), "global_pairs": world * nb, "lm_iterations_per_step": total_iters,
                           "batch_iters_per_s": total_iters / (ms_per_step * 1e-3), "precision": args.precision,
                           "nvalid_fraction_finest_level": nvalid_frac, "planted_motion": "4 deg / 8 cm" if args.motion == "large" else "1 deg / 2 cm",
                           "conv2_layout": "[F2|gx|gy] (3C channels, the reference's BundleIteration boundary)" if args.layout == "concat"
                                           else "F2 only (C channels); the kernel recomputes gx, gy on the fly (reference grad_fixed, bundlenet.py:92-100)",
                           "l2": "inputs (~33 GB/GPU) far exceed the 126 MB L2; no flush needed",
                           "parallelism": f"pairs sharded over {world} GPU(s), one all-gather of (R,T,W) per step"},
                "clocks": clocks, "e2e": e2e, "gpu_launches": args.steps * (1 + total_iters * 3), "precision_check": precision_check,
                "roofline": roofline, "cpu_baseline": cpu_baseline}
        print(json.dumps(line))
    if world > 1:
        td.destroy_process_group()


def run_e2e(args, sc, levels, packed, ws, world, local, dev, total_iters, prec):
    """The call a user with host-resident inputs makes.  Default: banet_b200.host_pipeline.ResizeHostSolver at the reference's BundleResize
    boundary; every step copies every input host->device and the result device->host (copies of later pair chunks overlap the solve)."""
    from banet_b200 import dist as bdist, synth
    from banet_b200.host_pipeline import HostSolver, ResizeHostSolver
    C = args.channels
    rank = int(os.environ.get("RANK", "0"))
    pin = lambda t: torch.empty(t.shape, dtype=t.dtype, device="cpu", pin_memory=True).copy_(t)
    if args.e2e_boundary == "resize":
        rs = synth.make_resize_scene(args.nb, H_FULL, W_FULL, C, args.bases, level_ids=LEVEL_IDS, seed=4321 + 1000 * rank, device=dev)
        solver = ResizeHostSolver([pin(l) for l in rs.layers], pin(rs.basis), pin(rs.init_depth), pin(rs.intr), rs.scales, chunks=args.e2e_chunks,
                                  device=dev, precision=prec)
        hR, hT, hW = pin(rs.R0), pin(rs.T0), pin(rs.W0)
        del rs
        torch.cuda.empty_cache()
        boundary = ("the reference's BundleResize boundary (bundlenet.py:332-399): feature pyramid of the image batch (pair b = images b, b+nb/2), half-resolution "
                    "basis and depth, intrinsics in pinned host memory; conv1 (zero copy), conv2 (F2 only), p, D, B derived on the device every step")
        api = f"banet_b200.host_pipeline.ResizeHostSolver(chunks={args.e2e_chunks}).solve"
    else:
        feat = args.e2e_boundary == "features" and args.layout == "concat"
        host = []
        for l in sc.levels:
            tens = {"grid": l.grid}
            for name in ("conv1", "conv2", "intr", "p", "D", "B"):
                t = getattr(l, name)
                if name == "conv2" and feat:
                    t = t[..., :C].contiguous()
                tens[name] = pin(t)
            host.append(tens)
        solver = HostSolver(host, derive_gradients=feat, chunks=args.e2e_chunks, device=dev, precision=prec)
        hR, hT, hW = pin(sc.R0), pin(sc.T0), pin(sc.W0)
        boundary = ("per-level tensors: feature maps (C channels) + conv1, p, D, B, intr in pinned host memory; [F2|gx|gy] derived on the device every step "
                    "(banet_grad_fixed_concat)") if feat else "every level tensor, conv2 as the 3C [F2|gx|gy] tensor, in pinned host memory"
        api = f"banet_b200.host_pipeline.HostSolver(chunks={args.e2e_chunks}).solve"
    h2d = solver.h2d_bytes + (hR.numel() + hT.numel() + hW.numel()) * 4
    oR = torch.empty_like(hR).pin_memory(); oT = torch.empty_like(hT).pin_memory(); oW = torch.empty_like(hW).pin_memory()
    d2h = (oR.numel() + oT.numel() + oW.numel()) * 4 * world
    last = {}

    def e2e_step():
        R, T, W, status = solver.solve(hR, hT, hW, args.iters, mlp_packed=packed, l2_regularizer_base=1000.0,
                                       out=None if world > 1 else (oR, oT, oW))
        last["status"] = status
        if world > 1:
            R, T, W = bdist.all_gather_solution(R, T, W)
            return R.cpu(), T.cpu(), W.cpu()
        torch.cuda.current_stream().synchronize()
        return oR, oT, oW

    e2e_step()
    torch.cuda.synchronize()
    bad_pairs = int((last["status"] != 0).sum())
    if world > 1:
        import torch.distributed as td
        td.barrier(device_ids=[local])
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.e2e_steps):
        e2e_step()
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if world > 1:
        tms = torch.tensor([ms], device=dev, dtype=torch.float64)
        td.all_reduce(tms, op=td.ReduceOp.MAX); ms = float(tms.item())
    per = ms / args.e2e_steps * 1e-3
    return {"value": world * args.nb * total_iters / per, "unit": UNIT, "h2d_bytes_per_step": h2d * world,
            "d2h_bytes_per_step": d2h, "ms_per_step": per * 1e3, "steps": args.e2e_steps, "boundary": boundary, "api": api,
            "pairs_with_skipped_steps": bad_pairs,
            "note": "pinned host -> device copy of every input + solve + device -> host of (R,T,W) per step; copies of later pair chunks overlap the "
                    "solve of the current one"}


if __name__ == "__main__":
    main()
